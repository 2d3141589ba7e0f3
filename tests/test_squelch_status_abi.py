"""The squelch reporting / threshold entry points refuse NULL handles before anything touches the device, also without
a GPU."""


def test_squelch_calls_refuse_null_handles():
    from sdrtrunk_b200 import native
    L = native.lib()
    assert L.sdrgpu_bank_set_squelch_reporting(None, 1) == native.ERR_INVALID_ARG
    assert L.sdrgpu_bank_set_squelch_reporting(None, 0) == native.ERR_INVALID_ARG
    assert L.sdrgpu_bank_set_squelch_threshold(None, 0, -40.0) == native.ERR_INVALID_ARG
    assert L.sdrgpu_bank_set_squelch_threshold(None, -1, float("nan")) == native.ERR_INVALID_ARG
    assert b"NULL" in L.sdrgpu_last_error()


def test_status_bits_match_the_oracle_codes():
    """the status byte's state codes are the oracle's PowerSquelch states (orc_filters.c SQ_*)"""
    import oracle
    from sdrtrunk_b200 import native
    fm = oracle.SquelchingFMDemodulator(0.01, -40.0, 4)
    assert fm.s.sq.state == native.SQUELCH_MUTE
    assert (native.SQUELCH_ATTACK, native.SQUELCH_DECAY, native.SQUELCH_UNMUTE) == (0, 1, 3)
    assert native.SQUELCH_CHANGED == 4
