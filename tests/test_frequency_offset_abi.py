"""sdrgpu_chan_set_frequency_offsets: exported, and its argument checks run before anything touches the device, also
without a GPU.  The refusals that need a live channelizer (out of range, listed twice, before the sample rate) and the
check that a refused call changes nothing are at the end, on the GPU."""
import ctypes as C

import numpy as np
import pytest


def _args(*values):
    idx = (C.c_int * max(len(values), 1))(*[i for i, _ in values])
    hz = (C.c_longlong * max(len(values), 1))(*[v for _, v in values])
    return idx, hz


def test_symbol_is_exported_with_a_prototype():
    from sdrtrunk_b200 import native
    lib = C.CDLL(native.LIB_PATH)
    assert hasattr(lib, "sdrgpu_chan_set_frequency_offsets")
    assert "sdrgpu_chan_set_frequency_offsets" in native.PROTOTYPES


def test_null_and_empty_arguments_are_refused():
    from sdrtrunk_b200 import native
    L = native.lib()
    idx, hz = _args((0, 100))
    assert L.sdrgpu_chan_set_frequency_offsets(None, idx, hz, 1) == native.ERR_INVALID_ARG
    assert b"NULL" in L.sdrgpu_last_error()
    fake = C.c_void_p(16)   # never dereferenced: the NULL / count checks come first
    assert L.sdrgpu_chan_set_frequency_offsets(fake, None, hz, 1) == native.ERR_INVALID_ARG
    assert L.sdrgpu_chan_set_frequency_offsets(fake, idx, None, 1) == native.ERR_INVALID_ARG
    assert L.sdrgpu_chan_set_frequency_offsets(fake, idx, hz, 0) == native.ERR_INVALID_ARG
    assert L.sdrgpu_chan_set_frequency_offsets(fake, idx, hz, -3) == native.ERR_INVALID_ARG


@pytest.mark.gpu
def test_refusals_on_a_live_channelizer_change_nothing(gpu):
    """out of range, listed twice and a nonzero offset before the sample rate are refused with their codes; the rows that
    follow equal those of a channelizer that was never given the refused calls, bit for bit"""
    import oracle
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    L = gpu.lib()
    m = 96
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    entries = [([3], 700), ([10, 11], -1500), ([40], 0), ([70], 2200)]
    x = np.random.default_rng(5).standard_normal(2 * 48 * 300).astype(np.float32) * 0.1

    def channelizer():
        ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
        ch.setOutputChannels(entries)
        return ch

    ref, ch = channelizer(), channelizer()
    want = [ref.receiveChannels(x[:2 * 48 * 100]), ref.receiveChannels(x[2 * 48 * 100:])]
    got = [ch.receiveChannels(x[:2 * 48 * 100])]
    for values, code in ((((4, 100),), gpu.ERR_INVALID_ARG), (((-1, 100),), gpu.ERR_INVALID_ARG),
                         (((0, 100), (2, 5), (0, 200)), gpu.ERR_INVALID_ARG),
                         (((0, 100), (4, 100)), gpu.ERR_INVALID_ARG)):
        idx, hz = _args(*values)
        assert L.sdrgpu_chan_set_frequency_offsets(ch._h, idx, hz, len(values)) == code, values
    got.append(ch.receiveChannels(x[2 * 48 * 100:]))
    for g, w in zip(got, want):
        assert np.array_equal(g, w)

    # before sdrgpu_chan_set_sample_rate: a nonzero offset is refused, a zero offset is fine
    h = C.c_void_p()
    t32 = np.ascontiguousarray(taps, np.float32)
    gpu.check(L.sdrgpu_chan_create(C.byref(h), t32.ctypes.data_as(C.POINTER(C.c_float)), t32.size, m, 1 << 16))
    idx, hz = _args((5, 300))
    assert L.sdrgpu_chan_set_frequency_offsets(h, idx, hz, 1) == gpu.ERR_BAD_STATE
    idx, hz = _args((5, 0))
    assert L.sdrgpu_chan_set_frequency_offsets(h, idx, hz, 1) == gpu.OK
    L.sdrgpu_chan_destroy(h)
