"""Pins the data and constants the reference embeds in its own sources (the only "golden vectors" it holds for this
path) against what the oracle and the product carry.  The reference's values are stored in
tests/golden/reference_constants.json: the MMSE table as tools/gen_mmse_table.py copied it from Interpolator.java, the
rest as they stand in the Java sources named beside each check."""
import json
import os
import re

import numpy as np

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_constants.json")))


def source(*path):
    return open(os.path.join(ROOT, *path)).read()


def test_mmse_interpolator_table_is_the_references():
    """dsp/filter/interpolator/Interpolator.java"""
    ref = np.array([[np.float32(v) for v in row.split()] for row in REF["mmse_interpolator_taps"]], np.float32)
    assert ref.shape == (129, 8)
    text = source("include", "sdr_mmse_taps.h")
    mine = np.array([np.float32(v[:-1]) for v in re.findall(r"[-+]?\d\.\d+e[-+]\d+f", text)], np.float32).reshape(129, 8)
    assert np.array_equal(mine, ref)


def test_window_and_envelope_constants():
    """dsp/filter/Window.java (Blackman a0..a2), sample/complex/Complex.java (envelope and fast normalisation),
    dsp/gain/ComplexFeedForwardGainControl.java (MINIMUM_ENVELOPE)"""
    a = [float(v) for v in REF["window_blackman_a"]]
    n = 23
    x = np.arange(n)
    want = a[0] - a[1] * np.cos(2 * np.pi * x / (n - 1)) + a[2] * np.cos(4 * np.pi * x / (n - 1))
    assert np.allclose(oracle.window("blackman", n), want, rtol=0, atol=1e-15)
    agc = REF["complex_feed_forward_gain_control"]
    weight, scalor = "%gf" % agc["envelope_minor_axis_weight"], "%gf" % REF["complex_fast_normalize_constant"]
    assert "(%s * qa)" % weight in source("oracle", "orc_filters.c")
    assert "__fmul_rn(%s, b)" % weight in source("sdrtrunk_b200", "csrc", "filters.cu")
    assert "(%s - norm)" % scalor in source("oracle", "orc_output.c")
    assert "__fsub_rn(%s, norm)" % scalor in source("sdrtrunk_b200", "csrc", "outputs.cu")
    floor = np.float32(agc["minimum_envelope"])
    y = oracle.agc_block(np.array([3e-5, -1e-5] * 1024, np.float32))          # envelope below the minimum: gain 1 / 1e-4
    assert np.array_equal(y[:2], np.array([3e-5, -1e-5], np.float32) * (np.float32(1.0) / floor))


def test_decoder_front_end_constants():
    """module/decode/p25/phase1/P25P1DecoderC4FM.java, P25P1DecoderLSM.java, phase2/P25P2DecoderHDQPSK.java,
    dmr/DMRDecoder.java (symbol rate, PLL bandwidth, SAMPLE_COUNTER_GAIN / SYMBOL_TIMING_GAIN), dsp/psk/pll/PLLBandwidth.java,
    dsp/psk/InterpolatingSampleBuffer.java, dsp/symbol/Dibit.java, dsp/filter/channelizer/PolyphaseChannelSource.java"""
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp.bank import Dibit, PLLBandwidth
    assert {b.name: b.value for b in PLLBandwidth} == REF["pll_bandwidth"]
    assert {d.name: d.value for d in Dibit} == REF["dibit"]
    deviation = "%gf" % REF["maximum_deviation_samples_per_symbol"]
    for src in (source("oracle", "orc_psk.c"), source("sdrtrunk_b200", "csrc", "psk.cu")):
        assert "sps * (1.0f + %s)" % deviation in src and "sps * (1.0f - %s)" % deviation in src
    # the presets of the C ABI carry the same numbers
    cfg = native.BankConfig()
    presets = {"c4fm": native.PRESET_P25_C4FM, "lsm": native.PRESET_P25_LSM, "hdqpsk": native.PRESET_P25_HDQPSK,
               "dmr": native.PRESET_DMR}
    for kind, want in REF["decoders"].items():
        native.check(native.lib().sdrgpu_bank_config_preset(cfg, presets[kind], 1, 50000.0, None, 0, 1024))
        assert cfg.symbol_rate == want["symbol_rate"], kind
        assert cfg.pll_bandwidth == REF["pll_bandwidth"][want["pll_bandwidth"]], kind
        assert abs(cfg.sample_counter_gain - want["sample_counter_gain"]) < 1e-7, kind
        assert 2 * cfg.block_size == REF["processed_buffer_sample_size"] and cfg.agc == 1


def test_half_band_stage_plan_is_the_references():
    """ComplexDecimateX{N}Filter stage lengths / windows (SURVEY a9): decimation by 2^k runs the X{2^k} filter's stage, then
    the X{2^(k-1)} one's, down to X2; the oracle (orc_filters.c) and the product (bank.cu) build the same cascade"""
    first = {int(r): (length, window) for r, (length, window) in REF["complex_decimate_filter"].items()}
    plan = {rate: [first[r] for r in (8, 4, 2) if r <= rate] for rate in first}
    assert plan == {2: [(63, "HAMMING")], 4: [(23, "BLACKMAN"), (63, "HAMMING")],
                    8: [(15, "BLACKMAN"), (23, "BLACKMAN"), (63, "HAMMING")]}
    for src in (source("oracle", "orc_filters.c"), source("sdrtrunk_b200", "csrc", "bank.cu")):
        stages = {int(r): (int(n), w) for r, n, w in
                  re.findall(r"if \(r == (\d+)\) \{ len = (\d+); win = \w+_(BLACKMAN|HAMMING); \}", src)}
        other = re.search(r"else \{ len = (\d+); win = \w+_(BLACKMAN|HAMMING); \}", src)
        stages[2] = (int(other.group(1)), other.group(2))
        assert re.search(r"for \(int r = [\w>-]+; r >= 2; r /= 2\)", src)
        assert {r: stages[r] for r in first} == first


def test_sync_patterns_and_detector_constants():
    """dsp/symbol/FrameSync.java patterns, match threshold, delay lengths and sync-loss lengths of the P25 sync detectors
    (P25P1SyncDetector, P25P2SyncDetector, P25P1DataUnitDetector, P25P2SuperFrameDetector), as carried by the oracle
    (orc_sync.c) and the product (SyncTraits in psk.cu)."""
    fs = {k: int(v, 16) for k, v in REF["frame_sync"].items()}
    det = REF["sync_detectors"]
    assert len(fs) == 8
    oracle_src, product_src = source("oracle", "orc_sync.c"), source("sdrtrunk_b200", "csrc", "psk.cu")
    for src in (oracle_src, product_src):
        mine = set(int(v, 16) for v in re.findall(r"0x([0-9A-Fa-f]{10,12})ull", src))
        assert set(fs.values()) <= mine
    assert "s->threshold = %d;" % det["match_threshold"] in oracle_src
    assert "kSyncMatchThreshold = %d;" % det["match_threshold"] in product_src
    p1, p2 = det["p25_phase1"], det["p25_phase2"]
    for n in (p1["sync_loss_bits"], p2["sync_loss_bits"]):
        assert "s->sync_loss_threshold = %d;" % n in oracle_src and "loss_bits = %d;" % n in product_src
    assert "sync_size = %d;" % p1["sync_bits"] in oracle_src and "sync_size = %d;" % p2["sync_bits"] in oracle_src
    assert "symbol_rate = %.1f;" % p1["symbol_rate"] in oracle_src and "symbol_rate = %.1f;" % p2["symbol_rate"] in oracle_src
    assert oracle.SyncDetector(oracle.SYNC_P25_PHASE1, 50000.0).delay == p1["data_unit_dibit_length"] - p1["sync_dibit_length"]
    assert oracle.SyncDetector(oracle.SYNC_P25_PHASE2, 50000.0).delay == p2["delay_dibits"]
    # the rotated patterns are the normal one with every dibit's constellation point turned by 90 / 180 degrees:
    # +1 (00) -> +3 (01) -> -3 (11) -> -1 (10) -> +1 going counter-clockwise
    ccw = {0: 1, 1: 3, 3: 2, 2: 0}
    for phase, bits in (("PHASE1", p1["sync_bits"]), ("PHASE2", p2["sync_bits"])):
        d = [(fs["P25_%s_NORMAL" % phase] >> (bits - 2 - 2 * k)) & 3 for k in range(bits // 2)]
        def rotate(seq, quarter_turns):
            for _ in range(quarter_turns):
                seq = [ccw[v] for v in seq]
            return seq
        def pack(seq):
            v = 0
            for x in seq:
                v = (v << 2) | x
            return v
        assert pack(rotate(d, 1)) == fs["P25_%s_ERROR_90_CCW" % phase]
        assert pack(rotate(d, 2)) == fs["P25_%s_ERROR_180" % phase]
        assert pack(rotate(d, 3)) == fs["P25_%s_ERROR_90_CW" % phase]
