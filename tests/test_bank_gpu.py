"""Parity of the CUDA per-channel banks (through the C ABI) against the oracle.

Bars (BASELINE.json north_star): filters / AGC are float32 arithmetic restated op for op -> bit-exact;
FM discriminator output 1e-4 relative RMS (double atan from CUDA's libm vs glibc's: both < 1 ulp in double, the
float results agree except on rare double-rounding ties); decoded DQPSK dibits bit-exact.
"""
import numpy as np
import pytest
import scipy.signal as ss

import oracle
import siggen as sg

pytestmark = pytest.mark.gpu

TOL = 1e-4


def c4fm_taps():
    """the taps P25P1DecoderC4FM designs (P25P1DecoderC4FM.java:136-148 through RemezFIRFilterDesigner), 72 taps"""
    return oracle.c4fm_baseband_taps()


def hdqpsk_taps():
    """P25P2DecoderHDQPSK.java:155-166, 154 taps"""
    return oracle.hdqpsk_baseband_taps()


def _noise(rng, c, n, scale=0.3):
    return (scale * rng.standard_normal((c, 2 * n))).astype(np.float32)


# ------------------------------------------------------------------------------------------------ filters
@pytest.mark.parametrize("n_taps", [1, 7, 45, 72, 154, 301])
def test_complex_fir_bit_exact(gpu, n_taps):
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(n_taps)
    taps = rng.standard_normal(n_taps).astype(np.float32) / n_taps
    c, n = 5, 3 * 1024
    x = _noise(rng, c, n)
    bank = Bank(c, 50000.0, fir_taps=taps, fir_gain=1.5, max_samples_per_call=n)
    got = bank.process(x)
    for k in range(c):
        want = oracle.ComplexFIR(taps, 1.5).filter(x[k])
        assert np.array_equal(got[k], want), k


def test_fir_streaming_ragged_calls(gpu):
    """history carried across calls; samples that do not fill a 1024-sample assembler buffer stay pending
    (ReusableComplexBufferAssembler.java:99-167)"""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(1)
    taps = c4fm_taps()
    c, n = 3, 6 * 1024
    x = _noise(rng, c, n)
    bank = Bank(c, 50000.0, fir_taps=taps, max_samples_per_call=4096)
    parts, pos = [], 0
    for step in (1000, 24, 0, 3000, 72, 2048):
        parts.append(bank.process(x[:, 2 * pos:2 * (pos + step)]))
        pos += step
    assert pos == n
    got = np.concatenate(parts, axis=1)
    assert got.shape == (c, 2 * n)
    for k in range(c):
        assert np.array_equal(got[k], oracle.ComplexFIR(taps).filter(x[k]))


@pytest.mark.parametrize("rate", [2, 4, 8, 16, 32, 64, 128, 256, 512, 1024])
def test_decimation_cascade_bit_exact(gpu, rate):
    """every rate DecimationFilterFactory.getComplexDecimationFilter offers (DecimationFilterFactory.java:36-104)"""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(rate)
    c, n = 4, max(4096, 4 * rate)
    x = _noise(rng, c, 2 * n)
    bank = Bank(c, 50000.0 * rate, decimation=rate, block_size=n, max_samples_per_call=n)
    got = np.concatenate([bank.process(x[:, :2 * n]), bank.process(x[:, 2 * n:])], axis=1)
    assert got.shape == (c, 2 * (2 * n // rate))
    for k in range(c):
        d = oracle.Decimator(rate)
        want = np.concatenate([d.decimate_complex(x[k, :2 * n]), d.decimate_complex(x[k, 2 * n:])])
        assert np.array_equal(got[k], want), k


def test_agc_block_bit_exact(gpu):
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(2)
    c, n = 6, 4 * 1024
    x = _noise(rng, c, n, 0.01)
    x[2, 2048:4096] = 0.0          # silent buffer: gain clamps at 1 / 1e-4
    x[3] *= 1e-5
    got = Bank(c, 50000.0, agc=True, max_samples_per_call=n).process(x)
    for k in range(c):
        want = np.concatenate([oracle.agc_block(x[k, 2048 * b:2048 * (b + 1)]) for b in range(4)])
        assert np.array_equal(got[k], want), k


@pytest.mark.parametrize("n_taps", [5, 8, 24, 72, 154, 301])
def test_fir_agc_whole_buffers_bit_exact(gpu, n_taps):
    """FIR + block AGC over whole 1024-sample assembler buffers -- the decoders' framing -- in calls of 1, 7, 2, 4 and 3
    buffers (odd and even tile counts per CTA).  Calls that are not throttled run fir_agc_split_kernel (per-warp windows,
    split-phase maximum exchange); calls held to 1 or 2 CTAs per SM ask for more shared memory than the window needs and
    run the general fir_agc_kernel.  The two kernels alternate on one bank: the history a kernel leaves is the history
    the other one starts from"""
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(100 + n_taps)
    taps = (rng.standard_normal(n_taps) / n_taps).astype(np.float32)
    c = 7
    # (samples, FIR CTAs per SM: 0 = not throttled)
    steps = ((1024, 0), (7 * 1024, 1), (1000, 0), (24, 2), (2 * 1024, 0), (4 * 1024, 2), (500, 0), (524, 1), (3 * 1024, 0))
    n = sum(step for step, _ in steps)
    x = _noise(rng, c, n, 0.05)
    x[1, 2 * 3000:2 * 6000] = 0.0     # silent buffers: the gain clamps at 1 / 1e-4
    x[2] *= 1e-6
    bank = Bank(c, 50000.0, fir_taps=taps, fir_gain=1.25, agc=True, max_samples_per_call=8 * 1024)
    lib = native.lib()
    # a small bank would get one buffer per CTA: ask for the large banks' launch shape (3 consecutive buffers per CTA)
    native.check(lib.sdrgpu_set_tuning(native.TUNE_FIR_TILES_PER_CTA, 3))
    try:
        parts, pos = [], 0
        for step, ctas in steps:
            native.check(lib.sdrgpu_set_tuning(native.TUNE_THROTTLE_ALWAYS, 1 if ctas else 0))
            native.check(lib.sdrgpu_set_tuning(native.TUNE_FIR_CTAS_PER_SM, ctas))
            parts.append(bank.process(x[:, 2 * pos:2 * (pos + step)]))
            pos += step
    finally:
        native.check(lib.sdrgpu_set_tuning(native.TUNE_FIR_TILES_PER_CTA, 0))
        native.check(lib.sdrgpu_set_tuning(native.TUNE_THROTTLE_ALWAYS, 0))
        native.check(lib.sdrgpu_set_tuning(native.TUNE_FIR_CTAS_PER_SM, 0))
    got = np.concatenate(parts, axis=1)
    assert got.shape == (c, 2 * n)
    for k in range(c):
        y = oracle.ComplexFIR(taps, 1.25).filter(x[k])
        want = np.concatenate([oracle.agc_block(y[2048 * b:2048 * (b + 1)]) for b in range(n // 1024)])
        assert np.array_equal(got[k], want), k


def test_single_channel_drop_in_classes(gpu):
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import (ComplexFeedForwardGainControl, ComplexFIRFilter2, DecimationFilterFactory,
                                   RealFIRFilter2)
    rng = np.random.default_rng(3)
    x = _noise(rng, 1, 2048)[0]
    taps = c4fm_taps()
    f = ComplexFIRFilter2(taps)
    ref = oracle.ComplexFIR(taps)
    for _ in range(2):
        assert np.array_equal(f.filter(x), ref.filter(x))
    r = rng.standard_normal(2000).astype(np.float32)
    assert np.array_equal(RealFIRFilter2(taps, 2.0).filter(r), oracle.RealFIR(taps, 2.0).filter(r))
    assert np.array_equal(ComplexFeedForwardGainControl(32).filter(x[:2048]), oracle.agc_block(x[:2048]))
    d = DecimationFilterFactory.getComplexDecimationFilter(4)
    assert np.array_equal(d.decimateComplex(x), oracle.Decimator(4).decimate_complex(x))
    rd = DecimationFilterFactory.getRealDecimationFilter(8)
    ref_rd = oracle.Decimator(8)
    for _ in range(2):
        assert np.array_equal(rd.decimateReal(r[:1600]), ref_rd.decimate_real(r[:1600]))
    with pytest.raises(native.IllegalArgumentException):
        DecimationFilterFactory.getComplexDecimationFilter(3)       # DecimationFilterFactory.java:62-64
    with pytest.raises(native.IllegalArgumentException):
        DecimationFilterFactory.getComplexDecimationFilter(8).decimateComplex(x[:24])   # ComplexDecimateX*Filter :47-54


# ------------------------------------------------------------------------------------------------ FM
def test_fm_demodulator_matches_oracle(gpu):
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(4)
    c, n = 4, 4096
    x = np.stack([sg.interleave(sg.nbfm(25000.0, 2 * n, audio_hz=400.0 * (k + 1), carrier_offset=100.0 * k) +
                                sg.awgn(rng, 2 * n, 1e-3)) for k in range(c)])
    x[1, 200:220] = 0.0            # inphase == 0 -> angle 0 branch (FMDemodulator.java:80-88)
    bank = Bank(c, 25000.0, demod=gpu.DEMOD_FM, fm_gain=1.0, block_size=n, max_samples_per_call=n)
    got = np.concatenate([bank.process(x[:, :2 * n]), bank.process(x[:, 2 * n:])], axis=1)
    exact = 0
    for k in range(c):
        want = oracle.FMDemodulator(1.0).demodulate(x[k])
        assert sg.rel_rms(got[k], want) < TOL
        assert np.max(np.abs(got[k] - want)) < 1e-6
        exact += int(np.sum(got[k] == want))
    assert exact > 0.999 * c * 2 * n      # in practice every sample is identical


def test_fm_wraps_like_atan(gpu):
    from sdrtrunk_b200.dsp import FMDemodulator
    z = np.exp(1j * np.cumsum(np.full(64, 2.0)))
    out = FMDemodulator(1.0).demodulate(sg.interleave(z))
    assert np.allclose(out[2:], 2.0 - np.pi, atol=1e-5)      # atan, not atan2 (FMDemodulator.java:85)
    assert out[0] == 0.0


def test_squelching_fm_matches_oracle(gpu):
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(5)
    n = 16 * 1024
    quiet = sg.awgn(rng, 4096, 1e-6)
    loud = sg.nbfm(25000.0, 6144, amplitude=0.5) + sg.awgn(rng, 6144, 1e-3)
    tail = sg.awgn(rng, n - 4096 - 6144, 1e-6)
    a = sg.interleave(np.concatenate([quiet, loud, tail]))
    b = sg.interleave(np.concatenate([loud, quiet, tail]))
    x = np.stack([a, b])
    # fast squelch (alpha 0.01) so that both the opening and the closing happen inside the test signal
    bank = Bank(2, 25000.0, demod=gpu.DEMOD_FM_SQUELCH, squelch_alpha=0.01, squelch_threshold_db=-40.0, squelch_ramp=4,
                block_size=2048, max_samples_per_call=n)
    got = np.concatenate([bank.process(x[:, :2 * 6144]), bank.process(x[:, 2 * 6144:])], axis=1)
    for k in range(2):
        want = oracle.SquelchingFMDemodulator(0.01, -40.0, 4).demodulate(x[k])
        assert np.array_equal(got[k] == 0.0, want == 0.0)        # identical gating
        assert np.any(want != 0.0) and np.any(want == 0.0)
        assert np.max(np.abs(got[k] - want)) < 1e-6


@pytest.mark.parametrize("rate", [0, 2, 4, 8])
def test_fused_nbfm_kernel_all_cascade_depths(gpu, rate):
    """nbfm_fused_kernel with no / one / two / three half-band stages (no decimation: the FIR reads the raw window;
    decimating: even / odd sample planes, skewed FIR input): 7 channels with different signals, squelch openings and
    closings, calls that end inside a tile and a FIR length that is not a multiple of 8 -- against the oracle's
    decimator -> ComplexFIR -> SquelchingFMDemodulator, buffer by buffer."""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(40 + rate)
    d = max(rate, 1)
    c, block = 7, 1024
    n = 11 * block                                    # channel-rate input samples per channel (11 assembler buffers)
    fir = oracle.nbfm_iq_taps() if rate != 4 else oracle.nbfm_iq_taps()[4:-4]     # 45 / 37 taps
    x = []
    for k in range(c):
        loud = sg.nbfm(25000.0 * d, n, audio_hz=300.0 * (k + 1), carrier_offset=150.0 * k, amplitude=0.3) + sg.awgn(rng, n, 1e-3)
        env = np.ones(n)
        env[(k * 997) % (n // 2):(k * 997) % (n // 2) + n // 4] = 1e-5          # a quiet stretch somewhere: squelch closes
        x.append(sg.interleave(loud * env))
    x = np.stack(x)
    bank = Bank(c, 25000.0 * d, demod=gpu.DEMOD_FM_SQUELCH, fir_taps=fir, decimation=rate, squelch_alpha=0.01,
                squelch_threshold_db=-40.0, squelch_ramp=4, block_size=block, max_samples_per_call=8 * block)
    cuts = [0, 3 * block, 4 * block, 9 * block, 11 * block]       # calls of 3, 1, 5 and 2 buffers
    got = np.concatenate([bank.process(x[:, 2 * a:2 * b]) for a, b in zip(cuts[:-1], cuts[1:])], axis=1)
    assert got.shape == (c, n // d)
    for k in range(c):
        dec = oracle.Decimator(rate) if rate else None
        f, fm = oracle.ComplexFIR(fir), oracle.SquelchingFMDemodulator(0.01, -40.0, 4)
        want = []
        for b in range(n // block):
            buf = x[k, 2 * block * b:2 * block * (b + 1)]
            want.append(fm.demodulate(f.filter(dec.decimate_complex(buf) if dec else buf)))
        want = np.concatenate(want)
        assert np.array_equal(got[k] == 0.0, want == 0.0), (rate, k)       # identical gating
        assert np.any(want != 0.0) and np.any(want == 0.0)
        assert np.max(np.abs(got[k] - want)) < 1e-6, (rate, k)
        assert np.mean(got[k] == want) > 0.999


@pytest.mark.parametrize("rate, agc", [(16, False), (32, False), (4, True)])
def test_five_kernel_nbfm_path(gpu, rate, agc):
    """FM banks that nbfm_fused_kernel does not fit: halfband_kernel stages, the FIR kernels, then squelch_gate_kernel,
    fm_kernel and fm_carry_kernel -- four half-band stages (decimation 16), an 11-tap first stage (decimation 32), and
    block AGC (512-sample AGC buffers) -- against the oracle's decimator -> ComplexFIR [-> AGC] -> SquelchingFMDemodulator,
    buffer by buffer.  Every channel has a quiet stretch of 1536 output samples: the squelch opens, closes and opens
    again at the output rate."""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(60 + rate)
    c, block = 3, 2048
    n = 4096 * rate                                   # channel-rate input samples per channel (4096 outputs)
    fir = oracle.nbfm_iq_taps()
    x = []
    for k in range(c):
        loud = sg.nbfm(25000.0 * rate, n, audio_hz=300.0 * (k + 1), carrier_offset=150.0 * k, amplitude=0.3) + sg.awgn(rng, n, 1e-3)
        env = np.ones(n)
        q0 = n // 8 + k * n // 16
        env[q0:q0 + 3 * n // 8] = 1e-7                # quiet enough to close the squelch behind the AGC's 1e4 gain too
        x.append(sg.interleave(loud * env))
    x = np.stack(x)
    bank = Bank(c, 25000.0 * rate, demod=gpu.DEMOD_FM_SQUELCH, fir_taps=fir, decimation=rate, agc=agc, squelch_alpha=0.01,
                squelch_threshold_db=-40.0, squelch_ramp=4, block_size=block, max_samples_per_call=n // 2)
    cuts = sorted({0, 3 * block, 4 * block, n // 2, n})
    got = np.concatenate([bank.process(x[:, 2 * a:2 * b]) for a, b in zip(cuts[:-1], cuts[1:])], axis=1)
    assert got.shape == (c, n // rate)
    for k in range(c):
        dec, f = oracle.Decimator(rate), oracle.ComplexFIR(fir)
        fm = oracle.SquelchingFMDemodulator(0.01, -40.0, 4)
        want = []
        for b in range(n // block):
            y = f.filter(dec.decimate_complex(x[k, 2 * block * b:2 * block * (b + 1)]))
            want.append(fm.demodulate(oracle.agc_block(y) if agc else y))
        want = np.concatenate(want)
        assert np.array_equal(got[k] == 0.0, want == 0.0), (rate, k)       # identical gating
        on = np.flatnonzero(want != 0.0)
        assert on.size and np.any(want[on[0]:] == 0.0), (rate, k)         # opens, then closes
        assert np.max(np.abs(got[k] - want)) < 1e-6, (rate, k)
        assert np.mean(got[k] == want) > 0.999


# ------------------------------------------------------------------------------------------------ DQPSK
def _p25_signal(kind, rng, n, k):
    rate = 6000.0 if kind == "hdqpsk" else 4800.0
    dib = rng.integers(0, 4, int(n * rate / 50000) + 8)
    off, tp = rng.uniform(-200, 200), rng.uniform(0, 1)
    if kind in ("c4fm", "dmr"):      # DMR is 4FSK at 4800 sym/s as well
        z = sg.c4fm(dib, carrier_offset=off, timing_phase=tp, n_samples=n)
    else:
        z = sg.dqpsk(dib, symbol_rate=rate, carrier_offset=off, timing_phase=tp, n_samples=n)
    return sg.interleave(z + sg.awgn(rng, n, 0.03)), dib


def _score(decoded, truth, skip=300):
    best = 0.0
    for lag in range(0, 24):
        n = min(decoded.size - lag, truth.size) - 20
        best = max(best, float(np.mean(decoded[lag + skip:lag + n] == truth[skip:n])))
    return best


def _preset(gpu, kind):
    return {"c4fm": (gpu.PRESET_P25_C4FM, oracle.C4FM, c4fm_taps()),
            "lsm": (gpu.PRESET_P25_LSM, oracle.LSM, None),
            "hdqpsk": (gpu.PRESET_P25_HDQPSK, oracle.HDQPSK, hdqpsk_taps()),
            "dmr": (gpu.PRESET_DMR, oracle.DMR, c4fm_taps())}[kind]


@pytest.mark.parametrize("lanes", [0, 8, 4, 2])
@pytest.mark.parametrize("kind", ["c4fm", "lsm", "hdqpsk", "dmr"])
def test_p25_bank_dibits_bit_exact(gpu, kind, lanes):
    """lanes = 8 / 4 / 2: psk_multi_kernel (several samples of a period per lane, 4 / 8 / 16 channels per warp)"""
    from sdrtrunk_b200.dsp import Bank
    preset, okind, taps = _preset(gpu, kind)
    rng = np.random.default_rng({"c4fm": 21, "lsm": 22, "hdqpsk": 23, "dmr": 24}[kind])
    c, n = 12, 20 * 1024
    sigs = [_p25_signal(kind, rng, n, k) for k in range(c)]
    x = np.stack([s[0] for s in sigs])
    x[5] *= 1e-3                                    # AGC brings a weak channel up
    bank = Bank.preset(preset, c, 50000.0, taps, max_samples_per_call=8 * 1024)
    bank.setDemodulatorLanes(lanes)
    parts = [bank.process(x[:, 2 * a:2 * b], want_filtered=True) for a, b in ((0, 8192), (8192, 9000), (9000, 17000), (17000, n))]
    for k in range(c):
        got = np.concatenate([p[0][k] for p in parts])
        agc = np.concatenate([p[1][k] for p in parts])
        want, want_agc = oracle.P25Chain(okind, 50000.0, taps).receive(x[k], want_agc=True)
        assert np.array_equal(agc, want_agc), k                      # filter + AGC tap point
        assert got.size == want.size, k
        assert np.array_equal(got, want), k                          # dibits bit-exact
        # and the decode is a real one: matches the transmitted dibits after acquisition
        assert _score(want, sigs[k][1]) > 0.98, k


def test_psk_loop_state_and_inversion(gpu):
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(6)
    n = 8 * 1024
    x, _ = _p25_signal("c4fm", rng, n, 0)
    bank = Bank(1, 50000.0, demod=gpu.DEMOD_DQPSK_DECISION, block_size=1024, symbol_rate=4800.0, pll_bandwidth=300.0,
                sample_counter_gain=0.3, max_samples_per_call=n)
    ref = oracle.PSKDemodulator(oracle.DECISION_DIRECTED, 50000.0, 4800.0, 300.0, 0.3)
    half = 2 * 4096
    a = bank.process(x[:half].reshape(1, -1))[0]
    assert np.array_equal(a, ref.receive(x[:half]))
    st, want = bank.loopState(0), ref.state()
    assert st[0] == want[0] and st[1] == want[1]               # double PLL state identical
    assert np.float32(st[2]) == np.float32(want[2]) and np.float32(st[3]) == np.float32(want[3])
    bank.correctInversion(0, np.pi / 2)                        # CostasLoop.correctInversion (:91-104)
    ref.correct_inversion(np.pi / 2)
    b = bank.process(x[half:].reshape(1, -1))[0]
    assert np.array_equal(b, ref.receive(x[half:]))
    assert bank.loopState(0)[1] == ref.state()[1]


def test_psk_drop_in_classes(gpu):
    from sdrtrunk_b200.dsp import (CostasLoop, DQPSKGardnerDemodulator, InterpolatingSampleBuffer, PLLBandwidth)
    rng = np.random.default_rng(7)
    x, _ = _p25_signal("lsm", rng, 4 * 2048, 0)
    pll = CostasLoop(50000.0, 4800.0)
    pll.setPLLBandwidth(PLLBandwidth.BW_200)
    demod = DQPSKGardnerDemodulator(pll, InterpolatingSampleBuffer(50000.0 / 4800.0, 0.3))
    seen = []
    demod.setSymbolListener(lambda d: seen.append(d.getValue()))
    ref = oracle.PSKDemodulator(oracle.GARDNER, 50000.0, 4800.0, 200.0, 0.3)
    want = []
    for b in range(4):
        buf = x[2 * 2048 * b:2 * 2048 * (b + 1)]
        demod.receive(buf)
        want.extend(ref.receive(buf).tolist())
    assert seen == want


def _sync_case(kind, rng, n, offset, with_sync=True):
    """a channel whose dibit stream carries the protocol's sync pattern every 180 symbols, at a carrier offset"""
    p2 = kind == "hdqpsk"
    rate = 6000.0 if p2 else 4800.0
    n_sym = int(n * rate / 50000) + 8
    pattern, bits = (sg.P25_PHASE2_SYNC, 40) if p2 else (sg.P25_PHASE1_SYNC, 48)
    dib = sg.dibits_with_sync(rng, n_sym, pattern, bits) if with_sync else rng.integers(0, 4, n_sym).astype(np.uint8)
    tp = rng.uniform(0, 1)
    if kind == "c4fm":
        z = sg.c4fm(dib, carrier_offset=offset, timing_phase=tp, n_samples=n, amplitude=0.5)
    else:
        z = sg.dqpsk(dib, symbol_rate=rate, carrier_offset=offset, timing_phase=tp, n_samples=n, amplitude=0.5)
    return sg.interleave(z + sg.awgn(rng, n, 0.01))


@pytest.mark.parametrize("kind,lanes", [("c4fm", 0), ("lsm", 0), ("hdqpsk", 0), ("c4fm", 16), ("hdqpsk", 16), ("lsm", 1),
                                        ("c4fm", 8), ("c4fm", 4), ("lsm", 8), ("lsm", 4), ("hdqpsk", 8), ("hdqpsk", 4),
                                        ("c4fm", 2), ("hdqpsk", 2)])
def test_sync_detector_and_inversion_feedback_on_device(gpu, kind, lanes):
    """SURVEY 8f #3: the framer's sync detector + PLLPhaseInversionDetector feedback run inside the demodulator
    kernel.  Channels locked 90 / 180 degrees off (carrier offset = +-rate/4, rate/2) must be corrected at the very
    symbol the reference corrects them: every byte (dibit | event << 2 | errors << 5) equals the oracle's."""
    from sdrtrunk_b200.dsp import Bank
    preset, okind, taps = _preset(gpu, kind)
    skind, okind_sync, rate = ((gpu.SYNC_P25_PHASE2, oracle.SYNC_P25_PHASE2, 6000.0) if kind == "hdqpsk"
                               else (gpu.SYNC_P25_PHASE1, oracle.SYNC_P25_PHASE1, 4800.0))
    rng = np.random.default_rng({"c4fm": 31, "lsm": 32, "hdqpsk": 33}[kind])
    n = 24 * 1024
    offsets = [0.0, rate / 4 - 50, -rate / 4 - 50, rate / 2 - 100, 120.0, -rate / 4 + 30, rate / 4, 0.0]
    x = np.stack([_sync_case(kind, rng, n, off, with_sync=(k != 7)) for k, off in enumerate(offsets)])
    bank = Bank.preset(preset, len(offsets), 50000.0, taps, max_samples_per_call=8 * 1024)
    bank.setDemodulatorLanes(lanes)
    bank.setSyncDetector(skind)
    parts = [bank.process(x[:, 2 * a:2 * b]) for a, b in ((0, 8192), (8192, 9000), (9000, 17000), (17000, n))]
    seen = set()
    for k in range(len(offsets)):
        got = np.concatenate([p[k] for p in parts])
        chain = oracle.P25Chain(okind, 50000.0, taps)
        chain.attach_sync(okind_sync, 50000.0)
        want = chain.receive(x[k])
        assert got.size == want.size, k
        assert np.array_equal(got, want), (k, np.nonzero(got != want)[0][:5])
        events = (want >> 2) & 7
        seen |= set(int(e) for e in events[events > 0])
        if k in (1, 2, 3):      # rotated pattern first, normal ones after the correction
            first = events[events > 0]
            assert first[0] in (gpu.SYNC_EVENT_INVERSION_90_CW, gpu.SYNC_EVENT_INVERSION_90_CCW, gpu.SYNC_EVENT_INVERSION_180), k
            assert np.all(first[1:] == gpu.SYNC_EVENT_SYNC) and first.size >= 8, k
    assert {gpu.SYNC_EVENT_SYNC, gpu.SYNC_EVENT_INVERSION_90_CW, gpu.SYNC_EVENT_INVERSION_90_CCW,
            gpu.SYNC_EVENT_INVERSION_180, gpu.SYNC_EVENT_LOST} <= seen
    # switching the detector off restores plain dibits; switching it on again starts from a fresh detector
    bank2 = Bank.preset(preset, 1, 50000.0, taps, max_samples_per_call=n)
    bank2.setSyncDetector(skind)
    bank2.setSyncDetector(gpu.SYNC_NONE)
    assert np.array_equal(bank2.process(x[:1])[0], oracle.P25Chain(okind, 50000.0, taps).receive(x[0]))
    with pytest.raises(gpu.IllegalArgumentException):
        bank2.setSyncDetector(7)


@pytest.mark.parametrize("kind,lanes,sync", [("c4fm", 0, False), ("c4fm", 4, False), ("c4fm", 32, True), ("c4fm", 4, True),
                                             ("lsm", 0, False), ("hdqpsk", 16, True), ("hdqpsk", 1, False),
                                             ("c4fm", 2, True), ("hdqpsk", 2, True)])
def test_symbol_tap_matches_the_instrumented_demodulator(gpu, kind, lanes, sync):
    """SURVEY section 5 / DQPSK*DemodulatorInstrumented: the per-symbol tap of one channel of a bank (complex symbol, samples
    per symbol, PLL frequency, sampling point, PLL error) equals the oracle demodulator's taps on the same FIR / AGC output,
    for every kernel family, with and without the sync detector's inversion feedback, across ragged calls and a tap moved
    to another channel; the bank's own dibits do not change."""
    from sdrtrunk_b200.dsp import Bank
    preset, okind, taps = _preset(gpu, kind)
    gardner, rate, bw, gain = {"c4fm": (False, 4800.0, 300.0, 0.3), "lsm": (True, 4800.0, 200.0, 0.3),
                               "hdqpsk": (True, 6000.0, 300.0, 0.1)}[kind]
    skind, okind_sync = ((gpu.SYNC_P25_PHASE2, oracle.SYNC_P25_PHASE2) if kind == "hdqpsk"
                         else (gpu.SYNC_P25_PHASE1, oracle.SYNC_P25_PHASE1))
    rng = np.random.default_rng(61)
    n = 12 * 1024
    offsets = [40.0, rate / 4 - 50, -80.0, rate / 2 - 100, 10.0]
    x = np.stack([_sync_case(kind, rng, n, off) for off in offsets])
    bank = Bank.preset(preset, len(offsets), 50000.0, taps, max_samples_per_call=8 * 1024)
    bank.setDemodulatorLanes(lanes)
    if sync:
        bank.setSyncDetector(skind)
    plain = Bank.preset(preset, len(offsets), 50000.0, taps, max_samples_per_call=8 * 1024)
    plain.setDemodulatorLanes(lanes)
    if sync:
        plain.setSyncDetector(skind)
    refs = []
    for _ in offsets:
        d = oracle.PSKDemodulator(oracle.GARDNER if gardner else oracle.DECISION_DIRECTED, 50000.0, rate, bw, gain)
        if sync:
            d.attach_sync(oracle.SyncDetector(okind_sync, 50000.0))
        refs.append(d)
    tapped = 1
    bank.setSymbolTap(tapped)
    for i, (a, b) in enumerate(((0, 4096), (4096, 5000), (5000, 9192), (9192, n))):
        if i == 2:
            tapped = 3
            bank.setSymbolTap(tapped)
        dib, filt = bank.process(x[:, 2 * a:2 * b], want_filtered=True)
        want_dib = plain.process(x[:, 2 * a:2 * b])
        tap = bank.symbolTap()
        for k in range(len(offsets)):
            assert np.array_equal(dib[k], want_dib[k]), (i, k)
            ref_dib, ref_tap = refs[k].receive(filt[k], want_taps=True)
            assert np.array_equal(dib[k], ref_dib), (i, k)
            if k == tapped:
                assert tap.shape == ref_tap.shape and (tap.shape[0] > 300 or i == 1), (i, tap.shape, ref_tap.shape)
                assert np.array_equal(tap[:, [0, 1, 2, 4, 5]], ref_tap[:, [0, 1, 2, 4, 5]]), i
                assert np.array_equal(tap[:, 3], ref_tap[:, 3]), i          # loop frequency: the same doubles
    hz = bank.symbolTap(sampleRate=50000.0)
    assert np.allclose(hz[:, 3], tap[:, 3] * 50000.0 / (2 * np.pi))
    bank.setSymbolTap(None)
    with pytest.raises(gpu.IllegalStateException):
        bank.symbolTap()


def _p2_channel(rng, n, offset, holes=()):
    """HDQPSK channel with the Phase 2 sync pattern every 180 symbols (every ISCH a sync ISCH), optional noise holes"""
    n_sym = int(n * 6000 / 50000) + 8
    dib = rng.integers(0, 4, n_sym).astype(np.uint8)
    s = sg.sync_dibits(sg.P25_PHASE2_SYNC, 40)
    for k in range(60, n_sym - 20, 180):
        dib[k:k + 20] = s
    z = sg.dqpsk(dib, symbol_rate=6000.0, carrier_offset=offset, timing_phase=rng.uniform(0, 1), n_samples=n, amplitude=0.5)
    z = z + sg.awgn(rng, n, 0.01)
    for a, ln in holes:
        z[a:a + ln] = sg.awgn(rng, ln, 0.3)
    return sg.interleave(z)


@pytest.mark.parametrize("lanes", [0, 16, 1])
def test_phase2_framing_on_device(gpu, lanes):
    """SDRGPU_SYNC_P25_PHASE2_FRAMED: the reference's whole Phase 2 framing (P25P2SuperFrameDetector: fragment sync
    state machine, sync-loss accounting, sync detector + PLL inversion feedback while unsynchronized) inside the
    demodulator kernel: every byte (dibit | events << 2) equals the oracle's, through ragged calls, on channels that
    lock rotated, lose the signal and re-acquire."""
    from sdrtrunk_b200.dsp import Bank
    preset, okind, taps = _preset(gpu, "hdqpsk")
    rng = np.random.default_rng(41)
    n = 40 * 1024
    cases = [(0.0, ()), (1450.0, ()), (-1550.0, ()), (2900.0, ()), (80.0, ((15000, 12000),)), (0.0, ((0, n),))]
    x = np.stack([_p2_channel(rng, n, off, holes) for off, holes in cases])
    bank = Bank.preset(preset, len(cases), 50000.0, taps, max_samples_per_call=16 * 1024)
    bank.setSyncDetector(gpu.SYNC_P25_PHASE2_FRAMED)
    bank.setDemodulatorLanes(lanes)
    cuts = (0, 16384, 17000, 30000, n)
    parts = [bank.process(x[:, 2 * a:2 * b]) for a, b in zip(cuts[:-1], cuts[1:])]
    seen = 0
    for k in range(len(cases)):
        got = np.concatenate([p[k] for p in parts])
        chain = oracle.P25Chain(okind, 50000.0, taps)
        chain.attach_sync(oracle.SYNC_P25_PHASE2_FRAMED, 50000.0)
        want = chain.receive(x[k])
        assert got.size == want.size, k
        assert np.array_equal(got, want), (k, np.nonzero(got != want)[0][:5])
        ev = want >> 2
        seen |= int(np.bitwise_or.reduce(ev))
        frag = np.nonzero(ev & gpu.P2_EVENT_FRAGMENT)[0]
        if k < 5:
            assert frag.size >= 4 and np.all(np.diff(frag) >= 720), k      # fragments every 720 dibits while in sync
        else:
            assert frag.size == 0                                         # noise never frames
        if k in (1, 2, 3):
            assert np.any(ev & gpu.P2_EVENT_INVERSION), k                  # locked rotated, corrected on the device
    assert seen & gpu.P2_EVENT_SYNC_LOSS and seen & gpu.P2_EVENT_SYNCHRONIZED


def test_phase2_framing_thread_per_channel_kernel(gpu):
    """the same through psk_wide_kernel (one thread per channel), 3072 channels"""
    from sdrtrunk_b200.dsp import Bank
    taps = hdqpsk_taps()
    rng = np.random.default_rng(42)
    n = 20 * 1024
    cases = [(0.0, ()), (1450.0, ()), (-1550.0, ()), (30.0, ((8000, 6000),))]
    base = np.stack([_p2_channel(rng, n, off, holes) for off, holes in cases])
    c = 3072
    x = np.tile(base, (c // len(cases), 1))
    bank = Bank.preset(gpu.PRESET_P25_HDQPSK, c, 50000.0, taps, max_samples_per_call=n)
    bank.setSyncDetector(gpu.SYNC_P25_PHASE2_FRAMED)
    bank.setDemodulatorLanes(1)
    got = bank.process(x[:, :2 * 9 * 1024])
    got2 = bank.process(x[:, 2 * 9 * 1024:])
    want = []
    for k in range(len(cases)):
        chain = oracle.P25Chain(oracle.HDQPSK, 50000.0, taps)
        chain.attach_sync(oracle.SYNC_P25_PHASE2_FRAMED, 50000.0)
        want.append(chain.receive(base[k]))
    assert all(np.any((w >> 2) & gpu.P2_EVENT_FRAGMENT) for w in want)
    for k in range(c):
        assert np.array_equal(np.concatenate([got[k], got2[k]]), want[k % len(cases)]), k


def test_sync_detector_thread_per_channel_kernel(gpu):
    """the same through psk_wide_kernel (one thread per channel): six distinct channels tiled over 3072"""
    from sdrtrunk_b200.dsp import Bank
    taps = c4fm_taps()
    rng = np.random.default_rng(34)
    n = 10 * 1024
    offsets = [0.0, 1150.0, -1250.0, 2300.0, 90.0, -60.0]
    base = np.stack([_sync_case("c4fm", rng, n, off) for off in offsets])
    c = 3072
    x = np.tile(base, (c // len(offsets), 1))
    bank = Bank.preset(gpu.PRESET_P25_C4FM, c, 50000.0, taps, max_samples_per_call=n)
    bank.setDemodulatorLanes(1)
    bank.setSyncDetector(gpu.SYNC_P25_PHASE1)
    got = bank.process(x[:, :2 * 6 * 1024])
    got2 = bank.process(x[:, 2 * 6 * 1024:])
    want = []
    for k in range(len(offsets)):
        chain = oracle.P25Chain(oracle.C4FM, 50000.0, taps)
        chain.attach_sync(oracle.SYNC_P25_PHASE1, 50000.0)
        want.append(chain.receive(base[k]))
    assert any(np.any(((w >> 2) & 7) >= 2) for w in want)
    for k in range(c):
        assert np.array_equal(np.concatenate([got[k], got2[k]]), want[k % len(offsets)]), k


def _scattered(c, distinct):
    """signal index of every bank row: neighbouring rows, rows 32 / 64 apart (a warp / a block later) and rows one
    kernel tile apart all carry different signals, so a demodulator or filter that reads another row's samples fails"""
    r = np.arange(c)
    return (r * 37 + (r // distinct) * 11 + (r // 1024) * 5) % distinct


@pytest.mark.parametrize("c,lanes", [(1024, 0), (3072, 0), (4608, 0), (321, 16), (97, 1), (64, 32), (1500, 8), (203, 8),
                                     (2100, 4), (77, 4), (333, 2)])
def test_many_channels(gpu, c, lanes):
    """BASELINE config 4 shape: >= 1000 channel-domain streams.  64 distinct HDQPSK signals (own dibits, carrier offset,
    timing phase and noise) are scattered over the rows and EVERY row is compared with the oracle's decode of the signal
    it carries.  By bank size the demodulator runs one warp per channel (1024), two channels per warp (3072) or one
    thread per channel (4608); the forced layouts use odd channel counts (a last warp with idle lanes)."""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(8)
    n, distinct = 4 * 1024, 64
    sigs = [_p25_signal("hdqpsk", rng, n, k)[0] for k in range(distinct)]
    which = _scattered(c, distinct)
    assert all(which[k] != which[k + 1] for k in range(c - 1)) and all(which[k] != which[k + 32] for k in range(c - 32))
    x = np.stack(sigs)[which]
    taps = hdqpsk_taps()
    bank = Bank.preset(gpu.PRESET_P25_HDQPSK, c, 50000.0, taps, max_samples_per_call=n)
    bank.setDemodulatorLanes(lanes)
    got = [np.concatenate(parts) for parts in zip(bank.process(x[:, :2 * 3072]), bank.process(x[:, 2 * 3072:]))]
    want = [oracle.P25Chain(oracle.HDQPSK, 50000.0, taps).receive(sig) for sig in sigs]
    assert len({w.tobytes() for w in want}) == distinct          # the decodes differ, so a swapped row is visible
    for k in range(c):
        assert np.array_equal(got[k], want[which[k]]), k


def test_demodulator_layout_can_change_between_calls(gpu):
    """the three kernel variants share the per-channel state: switching between calls changes nothing"""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(18)
    n = 8 * 1024
    sigs = [_p25_signal("c4fm", rng, n, k)[0] for k in range(5)]
    x = np.stack(sigs)
    taps = c4fm_taps()
    bank = Bank.preset(gpu.PRESET_P25_C4FM, 5, 50000.0, taps, max_samples_per_call=n)
    bank.setSyncDetector(gpu.SYNC_P25_PHASE2_FRAMED)      # the framer's state is layout independent as well
    parts = []
    for i, lanes in enumerate((32, 16, 1, 8, 32, 4, 0, 16)):
        bank.setDemodulatorLanes(lanes)
        parts.append(bank.process(x[:, 2 * 1024 * i:2 * 1024 * (i + 1)]))
    with pytest.raises(gpu.IllegalArgumentException):
        bank.setDemodulatorLanes(7)
    for k in range(5):
        chain = oracle.P25Chain(oracle.C4FM, 50000.0, taps)
        chain.attach_sync(oracle.SYNC_P25_PHASE2_FRAMED, 50000.0)
        assert np.array_equal(np.concatenate([p[k] for p in parts]), chain.receive(sigs[k])), k
    # the sync detectors keep layout-specific state: the layout has to be chosen before they are enabled
    bank.setSyncDetector(gpu.SYNC_P25_PHASE1)
    with pytest.raises(gpu.IllegalStateException):
        bank.setDemodulatorLanes(1)
    with pytest.raises(gpu.IllegalStateException):
        bank.setDemodulatorLanes(8)                         # (psk_multi_kernel's per-symbol matcher keeps the thread kernel's state)


# ------------------------------------------------------------------------------------------------ pipeline
def test_pipeline_channelizer_to_c4fm_bank(gpu):
    """BASELINE config 3 shape at a size the oracle finishes in seconds: M = 96 tuner stream whose bins carry C4FM,
    channelizer -> 72-tap FIR -> AGC -> decision-directed demodulator without a host round trip."""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, fs = 96, 2.4e6
    rng = np.random.default_rng(9)
    n_ch = 6 * 1024
    bins = [3, 17, 40, 60, 95]
    base = []
    for k in bins:
        dib = rng.integers(0, 4, int(n_ch * 4800 / 50000) + 8)
        base.append(sg.c4fm(dib, carrier_offset=rng.uniform(-200, 200), timing_phase=rng.uniform(0, 1), n_samples=n_ch,
                            amplitude=0.05))
    wide = sg.multiplex(base, bins, m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-3)
    x = sg.interleave(wide)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    fir = c4fm_taps()

    chan = ComplexPolyphaseChannelizerM2(taps, int(fs), m)
    chan.setChannels(bins)
    bank = Bank.preset(gpu.PRESET_P25_C4FM, len(bins), 50000.0, fir, max_samples_per_call=n_ch)
    pipe = Pipeline(chan, bank)
    cut = 2 * (n_ch * m // 2) // 3 // 2 * 2
    got = [np.concatenate(parts) for parts in zip(pipe.process(x[:cut]), pipe.process(x[cut:]))]

    # (1) bit-exact against the oracle chain fed the same channel I/Q (what the GPU channelizer produced)
    same_iq = ComplexPolyphaseChannelizerM2(taps, int(fs), m)
    same_iq.setChannels(bins)
    ch_iq = same_iq.receiveChannels(x)
    # (2) equal after acquisition against the full oracle chain (its own channelizer; FFT rounding differs)
    res = oracle.Channelizer(taps, m).receive(x)
    for i, k in enumerate(bins):
        want_same = oracle.P25Chain(oracle.C4FM, 50000.0, fir).receive(ch_iq[i][: n_ch * 2])
        assert np.array_equal(got[i], want_same), k
        y = oracle.OneChannelOutputProcessor(50000.0, k, float(m)).process(res)
        want_full = oracle.P25Chain(oracle.C4FM, 50000.0, fir).receive(y[: n_ch * 2])
        assert got[i].size == want_full.size
        assert np.array_equal(got[i][200:], want_full[200:]), k


@pytest.mark.parametrize("packed", [False, True])
def test_pipeline_from_airspy_native_buffers(gpu, packed):
    """Airspy raw buffers -> (unpack, DC removal, Hilbert) -> channelizer -> C4FM bank, all on the device and chunked
    through host buffers, equals the same pipeline fed the oracle converter's float I/Q."""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, fs = 96, 2.4e6
    rng = np.random.default_rng(19)
    n_ch = 4 * 1024
    n_real = 2 * (n_ch * m // 2)
    real = sg.airspy_real_signal(rng, n_real, [(25000.0 * 3 + 500, 0.2), (-25000.0 * 20, 0.1)], fs=2 * fs, noise=0.05)
    raw = sg.airspy_raw(real, packed)
    ref = oracle.AirspySampleConverter()
    ref.setSamplePacking(packed)
    iq = ref.convert(raw)
    taps, fir, bins = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps(), [3, 17, 76]

    def build(fmt):
        chan = ComplexPolyphaseChannelizerM2(taps, int(fs), m)
        chan.setChannels(bins)
        chan.setSampleFormat(fmt)
        bank = Bank.preset(gpu.PRESET_P25_C4FM, len(bins), 50000.0, fir, max_samples_per_call=n_ch)
        return Pipeline(chan, bank)

    want = build("f32").process(iq)
    pipe = build("airspy_packed" if packed else "airspy")
    values = raw if packed else raw.view("<u2")
    cut = (n_real // 3 // 2 * 2) * (3 if packed else 2) // 2          # an even number of samples into the stream
    got = [np.concatenate(parts) for parts in zip(pipe.process(values[:cut]), pipe.process(values[cut:]))]
    for a, b in zip(got, want):
        assert a.size == b.size and a.size > 300
        assert np.array_equal(a, b)


def test_config1_nbfm_chain(gpu):
    """BASELINE configs[0] / SURVEY 8d config 1: 2.4 MS/s -> channelizer M = 96 -> bin 4 (50 kHz) -> ComplexDecimateX2
    -> 25 kHz -> 45-tap low-pass -> squelching FM discriminator, fused on the device, against the oracle chain.
    Tolerances (north_star): 25 kHz I/Q and demodulated floats 1e-4 relative RMS."""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, fs = 96, 2.4e6
    rng = np.random.default_rng(1)
    n = 48 * 1024 * 6                                  # 6 assembler buffers of channel samples
    t = np.arange(n) / fs
    carrier = 0.5 * np.exp(1j * (2.5 * np.sin(2 * np.pi * 1000.0 * t) + 2 * np.pi * 100000.0 * t))   # +/-2.5 kHz dev.
    x = sg.interleave(carrier + sg.awgn(rng, n, 1e-3))
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    fir = oracle.nbfm_iq_taps()                        # NBFMDecoder.java:306-325, 45 taps

    def gpu_chain(demod):
        chan = ComplexPolyphaseChannelizerM2(taps, int(fs), m)
        chan.setChannels([4])
        if demod:
            bank = Bank.preset(gpu.PRESET_NBFM, 1, 50000.0, fir, max_samples_per_call=8192)
        else:
            bank = Bank(1, 50000.0, fir_taps=fir, decimation=2, max_samples_per_call=8192)
        assert bank.decimation == 2
        pipe = Pipeline(chan, bank)
        cut = x.size // 3 // 2 * 2
        return np.concatenate([pipe.process(x[:cut]), pipe.process(x[cut:])], axis=1)[0]

    res = oracle.Channelizer(taps, m).receive(x, mode="f64")
    y = oracle.OneChannelOutputProcessor(50000.0, 4, float(m)).process(res)
    dec, f, fm = oracle.Decimator(2), oracle.ComplexFIR(fir), oracle.SquelchingFMDemodulator(0.0004, -78.0, 4)
    iq25, audio = [], []
    for b in range(y.size // 2048):
        d = f.filter(dec.decimate_complex(y[2048 * b:2048 * (b + 1)]))
        iq25.append(d)
        audio.append(fm.demodulate(d))
    iq25, audio = np.concatenate(iq25), np.concatenate(audio)

    got_iq = gpu_chain(False)
    assert got_iq.shape == iq25.shape and sg.rel_rms(got_iq, iq25) < TOL
    got = gpu_chain(True)
    assert got.shape == audio.shape
    assert sg.rel_rms(got, audio) < TOL
    assert np.max(np.abs(got - audio)) < 1e-5
    # it is the 1 kHz tone at +/-2.5 kHz deviation: peak angle per 25 kHz sample = 2 pi 2500 / 25000
    assert abs(np.max(got[1000:]) - 2 * np.pi * 2500 / 25000) < 2e-2


# ------------------------------------------------------------------------------------------------ edge cases
def test_empty_short_and_oversized_calls(gpu):
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(41)
    taps = c4fm_taps()
    bank = Bank.preset(gpu.PRESET_P25_C4FM, 2, 50000.0, taps, max_samples_per_call=2048)
    assert [d.size for d in bank.process(np.zeros((2, 0), np.float32))] == [0, 0]          # empty buffer
    x, _ = _p25_signal("c4fm", rng, 4096, 0)
    x = np.stack([x, x])
    a = bank.process(x[:, :2 * 1000])                                                       # < one assembler buffer
    assert [d.size for d in a] == [0, 0]
    b = bank.process(x[:, 2 * 1000:2 * 2048])                                               # completes two buffers
    ref = oracle.P25Chain(oracle.C4FM, 50000.0, taps).receive(x[0, :2 * 2048])
    assert np.array_equal(b[0], ref) and np.array_equal(b[1], ref)
    with pytest.raises(gpu.OverflowError_):
        bank.process(np.zeros((2, 2 * 4096), np.float32))                                   # > max_samples_per_call
    with pytest.raises(gpu.IllegalArgumentException):
        Bank(1, 50000.0, decimation=3)                                                      # DecimationFilterFactory.java:62-64
    with pytest.raises(gpu.IllegalArgumentException):
        Bank(1, 9000.0, demod=gpu.DEMOD_DQPSK_DECISION, symbol_rate=4800.0, pll_bandwidth=300.0,
             sample_counter_gain=0.3)                                                       # sample rate <= 2 * symbol rate


def test_pack_dibits_matches_oracle(gpu):
    import ctypes as C
    rng = np.random.default_rng(42)
    for n in (0, 1, 3, 4, 5, 103):
        d = rng.integers(0, 4, n).astype(np.uint8)
        out = np.zeros(n // 4 + 1, np.uint8)
        got = gpu.lib().sdrgpu_pack_dibits(d.ctypes.data_as(C.POINTER(C.c_uint8)), n, out.ctypes.data_as(C.POINTER(C.c_uint8)))
        want = oracle.pack_dibits(d)
        assert got == want.size and np.array_equal(out[:got], want)


def test_pipeline_result_is_independent_of_chunking_and_memory_space(gpu):
    """the time-chunked, stream-overlapped host path, the single pass and device-resident input give identical dibits"""
    import ctypes as C
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 16 * 1024
    rng = np.random.default_rng(43)
    bins = [2, 30, 77]
    base = [sg.c4fm(rng.integers(0, 4, int(n_ch * 0.096) + 8), carrier_offset=rng.uniform(-200, 200),
                    timing_phase=rng.uniform(0, 1), n_samples=n_ch, amplitude=0.05) for _ in bins]
    x = sg.interleave(sg.multiplex(base, bins, m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-3))
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()

    def run(chunks, device_input):
        chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
        chan.setChannels(bins)
        pipe = Pipeline(chan, Bank.preset(gpu.PRESET_P25_C4FM, len(bins), 50000.0, fir, max_samples_per_call=n_ch))
        pipe.setChunks(chunks)
        if not device_input:
            return pipe.process(x)
        L = gpu.lib()
        d_in = C.c_void_p()
        gpu.check(L.sdrgpu_device_alloc(C.byref(d_in), x.nbytes))
        gpu.check(L.sdrgpu_memcpy(d_in, gpu.ptr(x), x.nbytes, gpu.DEVICE, gpu.HOST))
        out = pipe.process(d_in.value, gpu.DEVICE, x.size)
        L.sdrgpu_device_free(d_in)
        return out

    ref = run(1, False)
    assert all(r.size > 1500 for r in ref)
    for chunks, dev in ((8, False), (3, False), (1, True), (8, True)):
        got = run(chunks, dev)
        assert all(np.array_equal(g, r) for g, r in zip(got, ref)), (chunks, dev)


def test_pipeline_call_with_more_chunks_than_an_int_has_bits(gpu):
    """a long host call cut into many small time chunks: the doubling ramp of leading chunk sizes must stop at the chunk
    size (it once overflowed after 21 doublings and the call never returned); the dibits equal the single pass"""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 40 * 1024
    rng = np.random.default_rng(46)
    bins = [11]
    base = [sg.c4fm(rng.integers(0, 4, int(n_ch * 0.096) + 8), carrier_offset=120.0, timing_phase=0.4, n_samples=n_ch,
                    amplitude=0.05)]
    x = sg.interleave(sg.multiplex(base, bins, m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-3))
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    out = []
    for chunks in (1, 64):
        chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
        chan.setChannels(bins)
        pipe = Pipeline(chan, Bank.preset(gpu.PRESET_P25_C4FM, len(bins), 50000.0, fir, max_samples_per_call=n_ch))
        pipe.setChunks(chunks)
        out.append(pipe.process(x)[0])
    assert out[0].size > 3500 and np.array_equal(out[0], out[1])


def test_config3_shape_all_400_channels(gpu):
    """BASELINE configs[2] at full width: 10 MS/s, M = 400, every bin carries C4FM; all 400 channels through the fused
    pipeline.  Every channel must decode its transmitted dibits (size-independent property), and a sample of channels
    is bit-exact against the oracle chain fed the same channel I/Q."""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 400, 8 * 1024
    rng = np.random.default_rng(44)
    dibs = [rng.integers(0, 4, int(n_ch * 0.096) + 8) for _ in range(m)]
    base = [sg.c4fm(dibs[k], carrier_offset=rng.uniform(-200, 200), timing_phase=rng.uniform(0, 1), n_samples=n_ch,
                    amplitude=0.02, phase0=rng.uniform(0, 6.28)) for k in range(m)]
    x = sg.interleave(sg.multiplex(base, list(range(m)), m, n_ch) + sg.awgn(rng, n_ch * m // 2, 2e-3))
    fir = c4fm_taps()
    chan = ComplexPolyphaseChannelizerM2(1e7, 9, maxInputFloats=x.size)
    pipe = Pipeline(chan, Bank.preset(gpu.PRESET_P25_C4FM, m, 50000.0, fir, max_samples_per_call=n_ch))
    got = pipe.process(x)
    assert len(got) == m
    scores = np.array([_score(got[k], dibs[k], skip=200) for k in range(m)])
    assert np.mean(scores > 0.97) > 0.95, np.sort(scores)[:10]
    slow = [int(k) for k in np.nonzero(scores <= 0.97)[0]]     # slow acquisitions are the algorithm's, not the port's:
    iq = ComplexPolyphaseChannelizerM2(1e7, 9, maxInputFloats=x.size).receiveChannels(x)
    for k in [0, 1, 199, 200, 201, 399] + slow:                # ... they must match the oracle bit for bit as well
        want = oracle.P25Chain(oracle.C4FM, 50000.0, fir).receive(iq[k])
        assert np.array_equal(got[k], want), k


def test_handles_are_independent_across_host_threads(gpu):
    """include/sdrgpu.h: one host thread <-> one handle <-> one CUDA stream; different handles are fully concurrent.
    Four pipelines run from four threads at once and each must reproduce the single-threaded result; handles are
    created and destroyed repeatedly (no state leaks between them)."""
    import threading
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 4 * 1024
    rng = np.random.default_rng(45)
    bins = [5, 60]
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    inputs = []
    for _ in range(4):
        base = [sg.c4fm(rng.integers(0, 4, int(n_ch * 0.096) + 8), carrier_offset=rng.uniform(-200, 200),
                        timing_phase=rng.uniform(0, 1), n_samples=n_ch, amplitude=0.05) for _ in bins]
        inputs.append(sg.interleave(sg.multiplex(base, bins, m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-3)))

    def run(x):
        chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
        chan.setChannels(bins)
        bank = Bank.preset(gpu.PRESET_P25_C4FM, len(bins), 50000.0, fir, max_samples_per_call=n_ch)
        pipe = Pipeline(chan, bank)
        half = x.size // 2 // 2 * 2
        out = [np.concatenate(p) for p in zip(pipe.process(x[:half]), pipe.process(x[half:]))]
        pipe.dispose()
        bank.dispose()
        chan.dispose()
        return out

    want = [run(x) for x in inputs]
    for _ in range(3):
        got = [None] * 4
        ths = [threading.Thread(target=lambda i=i: got.__setitem__(i, run(inputs[i]))) for i in range(4)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        for i in range(4):
            assert all(np.array_equal(a, b) for a, b in zip(got[i], want[i])), i


# ------------------------------------------------------------------------------------------------ several tuners, one bank
def _tuner_stream(rng, m, n_ch, bins, kind="c4fm"):
    base = [sg.c4fm(rng.integers(0, 4, int(n_ch * 0.096) + 8), carrier_offset=rng.uniform(-200, 200),
                    timing_phase=rng.uniform(0, 1), n_samples=n_ch, amplitude=0.05) for _ in bins]
    return sg.interleave(sg.multiplex(base, bins, m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-3))


@pytest.mark.parametrize("fmt", ["f32", "s8"])
def test_multi_tuner_pipeline_equals_single_tuner_pipelines(gpu, fmt):
    """sdrgpu_pipeline_create_multi: three tuners' channelizers feed consecutive row ranges of one bank; the dibits of
    every row equal those of three separate single-tuner pipelines (and so the oracle's), for the chunked host path, the
    single pass, device-resident input with and without time chunks, and ragged calls."""
    import ctypes as C
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 12 * 1024
    rng = np.random.default_rng(71)
    bins = [[2, 30, 77], [5, 6], [0, 47, 48, 95]]
    xs = [_tuner_stream(rng, m, n_ch, b) for b in bins]
    if fmt == "s8":
        xs = [np.clip(np.round(x * 128.0 * 4), -128, 127).astype(np.int8) for x in xs]
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    rows = sum(len(b) for b in bins)

    def chan_for(k):
        ch = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=xs[0].size)
        ch.setChannels(bins[k])
        ch.setSampleFormat(fmt)
        return ch

    want = []
    for k in range(3):
        pipe = Pipeline(chan_for(k), Bank.preset(gpu.PRESET_P25_C4FM, len(bins[k]), 50000.0, fir, max_samples_per_call=n_ch))
        pipe.setChunks(1)
        want += pipe.process(xs[k])
    assert len(want) == rows and all(w.size > 1000 for w in want)
    if fmt == "f32":   # ... and the single-tuner reference is the oracle's decode of the same channel I/Q
        iq = chan_for(1).receiveChannels(xs[1])
        assert np.array_equal(want[3], oracle.P25Chain(oracle.C4FM, 50000.0, fir).receive(iq[0]))

    def multi(chunks, device_chunks=1, device_input=False, cuts=()):
        pipe = Pipeline([chan_for(k) for k in range(3)], Bank.preset(gpu.PRESET_P25_C4FM, rows, 50000.0, fir,
                                                                     max_samples_per_call=n_ch))
        pipe.setChunks(chunks)
        pipe.setDeviceChunks(device_chunks)
        edges = [0] + [c // 2 * 2 for c in cuts] + [xs[0].size]
        parts = []
        for a, b in zip(edges[:-1], edges[1:]):
            seg = [x[a:b] for x in xs]
            if not device_input:
                parts.append(pipe.process(seg))
                continue
            L = gpu.lib()
            ptrs = []
            for s_ in seg:
                d = C.c_void_p()
                gpu.check(L.sdrgpu_device_alloc(C.byref(d), max(s_.nbytes, 16)))
                gpu.check(L.sdrgpu_memcpy(d, gpu.ptr(np.ascontiguousarray(s_)), s_.nbytes, gpu.DEVICE, gpu.HOST))
                ptrs.append(d)
            parts.append(pipe.process([d.value for d in ptrs], gpu.DEVICE, seg[0].size))
            for d in ptrs:
                L.sdrgpu_device_free(d)
        return [np.concatenate(p) for p in zip(*parts)]

    for kw in (dict(chunks=8), dict(chunks=1), dict(chunks=3, cuts=(xs[0].size // 3, xs[0].size // 3 + 4000)),
               dict(chunks=1, device_input=True), dict(chunks=1, device_chunks=4, device_input=True)):
        got = multi(**kw)
        assert len(got) == rows
        for r in range(rows):
            assert np.array_equal(got[r], want[r]), (kw, r)


@pytest.mark.parametrize("fmt", ["f32", "s8"])
def test_asynchronous_pipeline_calls_equal_the_synchronous_sequence(gpu, fmt):
    """sdrgpu_pipeline_submit_multi / sdrgpu_pipeline_wait: a stream of host buffers with two calls in flight (the H2D
    copies of call k + 1 overlap the kernels of call k; alternating staging buffers) gives every channel the dibits of
    the same buffers through synchronous calls -- calls long enough to be cut into chunks (left in flight), one too
    short for that (runs to completion inside submit), an empty one; then a synchronous call continues the stream."""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 40 * 1024
    rng = np.random.default_rng(91)
    bins = [[2, 30, 77], [5, 6, 95]]
    xs = [_tuner_stream(rng, m, n_ch, b) for b in bins]
    if fmt == "s8":
        xs = [np.clip(np.round(x * 128.0 * 4), -128, 127).astype(np.int8) for x in xs]
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    rows = sum(len(b) for b in bins)
    unit = m * 1024          # input values per assembler buffer of every channel
    sizes = [9 * unit, 11 * unit + 4000, 0, 1 * unit, 8 * unit, 6 * unit]
    sizes.append(xs[0].size - sum(sizes))
    assert sizes[-1] > 3 * unit
    edges = np.cumsum([0] + sizes)

    def pipeline():
        chans = []
        for k in range(2):
            ch = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=12 * unit)
            ch.setChannels(bins[k])
            ch.setSampleFormat(fmt)
            chans.append(ch)
        pipe = Pipeline(chans, Bank.preset(gpu.PRESET_P25_C4FM, rows, 50000.0, fir, max_samples_per_call=12 * 1024))
        pipe.setChunks(4)
        return pipe

    sync = pipeline()
    want = [sync.process([x[a:b] for x in xs]) for a, b in zip(edges[:-1], edges[1:])]
    assert sum(w.size for w in want[0]) > 1000

    pipe = pipeline()
    got = []
    for i, (a, b) in enumerate(zip(edges[:-2], edges[1:-1])):
        pipe.submit([x[a:b].copy() for x in xs])
        if i >= 1:
            got.append(pipe.wait())          # two in flight, then the oldest comes back
    got.append(pipe.wait())
    assert pipe.wait() is None
    got.append(pipe.process([x[edges[-2]:edges[-1]] for x in xs]))   # a synchronous call carries on from there
    assert len(got) == len(want)
    for i in range(len(want)):
        for r in range(rows):
            assert np.array_equal(got[i][r], want[i][r]), (i, r)

    # three submits without a wait, and a synchronous call with calls in flight, are refused
    pipe2 = pipeline()
    pipe2.submit([x[:9 * unit] for x in xs])
    pipe2.submit([x[9 * unit:18 * unit] for x in xs])
    with pytest.raises(gpu.IllegalStateException):
        pipe2.submit([x[18 * unit:27 * unit] for x in xs])
    with pytest.raises(gpu.IllegalStateException):
        pipe2.process([x[18 * unit:27 * unit] for x in xs])
    pipe2.wait()
    pipe2.wait()


def test_asynchronous_pipeline_random_call_sizes(gpu):
    """a longer stream through submit / wait with random call sizes (whole buffers, ragged, shorter than a chunk, empty),
    waits taken late or early (one or two calls in flight), 8-bit tuner samples: every call's dibits equal the synchronous
    sequence's -- the ordering of the two calls' copies, kernels and staging is by events only"""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 96 * 1024
    rng = np.random.default_rng(131)
    bins = [[1, 40], [9, 90]]
    xs = [np.clip(np.round(_tuner_stream(rng, m, n_ch, b) * 128.0 * 4), -128, 127).astype(np.int8) for b in bins]
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    rows = 4
    unit = m * 1024
    sizes, left = [], xs[0].size
    while left > 0:
        kind = rng.integers(0, 5)
        n = [int(rng.integers(2, 9)) * unit, int(rng.integers(1, 8 * unit // 2)) * 2, unit // 2, 0, 8 * unit][kind]
        n = min(n, left)
        sizes.append(n)
        left -= n
    edges = np.cumsum([0] + sizes)

    def pipeline():
        chans = []
        for k in range(2):
            ch = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=8 * unit)
            ch.setChannels(bins[k])
            ch.setSampleFormat("s8")
            chans.append(ch)
        pipe = Pipeline(chans, Bank.preset(gpu.PRESET_P25_C4FM, rows, 50000.0, fir, max_samples_per_call=9 * 1024))
        pipe.setChunks(3)
        pipe.setDeviceChunks(2)
        return pipe

    sync = pipeline()
    want = [sync.process([x[a:b] for x in xs]) for a, b in zip(edges[:-1], edges[1:])]
    pipe = pipeline()
    got, in_flight = [], 0
    for a, b in zip(edges[:-1], edges[1:]):
        if in_flight == 2 or (in_flight == 1 and rng.integers(0, 2)):
            got.append(pipe.wait())
            in_flight -= 1
        pipe.submit([x[a:b].copy() for x in xs])
        in_flight += 1
    while in_flight:
        got.append(pipe.wait())
        in_flight -= 1
    assert len(got) == len(want) and len(want) > 12
    for i in range(len(want)):
        for r in range(rows):
            assert np.array_equal(got[i][r], want[i][r]), (i, r, sizes[i])


def test_frequency_corrected_channels_through_the_filters_first_and_asynchronous_schedules(gpu):
    """Frequency-corrected channels in a two-tuner pipeline: the filters-first schedule (device-resident input, and the
    asynchronous stream built on it) launches the oscillator producers at the START of a call, two calls ahead
    (chan_osc_ahead, two-call rings), where the single-pass call tops its ring up behind the channelizer.  Every row's
    dibits must be the same through all three, over calls of different lengths that wrap the rings."""
    import ctypes as C
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 30 * 1024
    rng = np.random.default_rng(97)
    bins = [[2, 30, 77], [5, 6, 95]]
    offsets = [[37, -53, 120], [-200, 9, 64]]
    xs = [_tuner_stream(rng, m, n_ch, b) for b in bins]
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    rows = sum(len(b) for b in bins)
    unit = m * 1024
    sizes = [6 * unit, 8 * unit, 3 * unit, 8 * unit]
    sizes.append(xs[0].size - sum(sizes))
    edges = np.cumsum([0] + sizes)

    def pipeline(device_chunks):
        chans = []
        for k in range(2):
            ch = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=8 * unit)
            ch.setOutputChannels([([b], off) for b, off in zip(bins[k], offsets[k])])
            chans.append(ch)
        pipe = Pipeline(chans, Bank.preset(gpu.PRESET_P25_C4FM, rows, 50000.0, fir, max_samples_per_call=9 * 1024))
        pipe.setChunks(1)
        pipe.setDeviceChunks(device_chunks)
        return pipe

    single = pipeline(1)
    want = [single.process([x[a:b] for x in xs]) for a, b in zip(edges[:-1], edges[1:])]
    assert sum(w.size for w in want[1]) > 1000

    first = pipeline(2)          # device-resident input, two time chunks: the filters-first schedule
    L = gpu.lib()
    for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
        ptrs = []
        for x in xs:
            seg = np.ascontiguousarray(x[a:b])
            d = C.c_void_p()
            gpu.check(L.sdrgpu_device_alloc(C.byref(d), max(seg.nbytes, 16)))
            gpu.check(L.sdrgpu_memcpy(d, gpu.ptr(seg), seg.nbytes, gpu.DEVICE, gpu.HOST))
            ptrs.append(d)
        got = first.process([d.value for d in ptrs], gpu.DEVICE, int(b - a))
        for d in ptrs:
            L.sdrgpu_device_free(d)
        for r in range(rows):
            assert np.array_equal(got[r], want[i][r]), ("filters-first", i, r)

    stream = pipeline(2)
    got = []
    for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
        stream.submit([x[a:b].copy() for x in xs])
        if i >= 1:
            got.append(stream.wait())
    got.append(stream.wait())
    for i in range(len(want)):
        for r in range(rows):
            assert np.array_equal(got[i][r], want[i][r]), ("stream", i, r)


def test_multi_tuner_pipeline_argument_checks(gpu):
    import ctypes as C
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    taps, fir = oracle.sinc_m2_channelizer(25000.0, 96, 9), c4fm_taps()
    a = ComplexPolyphaseChannelizerM2(taps, 2400000, 96, maxInputFloats=96 * 2048)
    b = ComplexPolyphaseChannelizerM2(taps, 2400000, 96, maxInputFloats=96 * 2048)
    a.setChannels([1, 2])
    b.setChannels([3])
    with pytest.raises(gpu.IllegalArgumentException):      # 3 rows selected, bank has 4
        Pipeline([a, b], Bank.preset(gpu.PRESET_P25_C4FM, 4, 50000.0, fir, max_samples_per_call=2048))
    other = ComplexPolyphaseChannelizerM2(oracle.sinc_m2_channelizer(25000.0, 80, 9), 2000000, 80)
    other.setChannels([3])
    with pytest.raises(gpu.IllegalArgumentException):      # different channel counts cannot share a bank
        Pipeline([a, other], Bank.preset(gpu.PRESET_P25_C4FM, 3, 50000.0, fir, max_samples_per_call=2048))
    pipe = Pipeline([a, b], Bank.preset(gpu.PRESET_P25_C4FM, 3, 50000.0, fir, max_samples_per_call=2048))
    x = np.zeros(96 * 1024, np.float32)
    a.receiveChannels(x[:90])                               # tuner a is now 45 samples ahead of tuner b
    with pytest.raises(gpu.IllegalStateException):
        pipe.process([x, x])


def test_pipeline_oversized_and_null_input_is_rejected_before_any_copy(gpu):
    """ADVICE r1: the chunked host path drives the channelizer internals directly, so it has to make sdrgpu_chan_process's
    checks itself: a bank sized larger than the channelizer's max_input_floats must give OVERFLOW, not a copy past the
    end of the channelizer's staging."""
    import ctypes as C
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m = 96
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=2 * 48 * 2048)     # 2048 blocks per call
    chan.setChannels([4, 9])
    pipe = Pipeline(chan, Bank.preset(gpu.PRESET_P25_C4FM, 2, 50000.0, fir, max_samples_per_call=16 * 1024))
    pipe.setChunks(8)
    big = np.zeros(2 * 48 * 8192, np.float32)
    with pytest.raises(gpu.OverflowError_):
        pipe.process(big)
    L = gpu.lib()
    counts = np.zeros(2, np.int32)
    sym = np.zeros((2, 4096), np.uint8)
    st = L.sdrgpu_pipeline_process(pipe._h, None, 2 * 48 * 2048, gpu.HOST, gpu.ptr(sym), 4096, None, 0, gpu.ptr(counts), gpu.HOST)
    assert st == gpu.ERR_INVALID_ARG
    # the handle is still usable and in its reset state
    x = _tuner_stream(np.random.default_rng(5), m, 2048, [4, 9])
    got = pipe.process(x)
    ref = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
    ref.setChannels([4, 9])
    iq = ref.receiveChannels(x)
    for k in range(2):
        assert np.array_equal(got[k], oracle.P25Chain(oracle.C4FM, 50000.0, fir).receive(iq[k]))


def test_pipeline_host_input_device_output_does_not_keep_the_caller_pointer(gpu):
    """ADVICE r1: sdrgpu.h promises that no caller pointer is kept after a call returns.  Chunked path, pinned host input,
    DEVICE outputs: the input buffer is overwritten the moment the call returns, and the result must still be the one of
    the original samples."""
    import ctypes as C
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 16 * 1024
    rng = np.random.default_rng(73)
    bins = [2, 30, 77]
    x = _tuner_stream(rng, m, n_ch, bins)
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    L = gpu.lib()

    def build():
        chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
        chan.setChannels(bins)
        pipe = Pipeline(chan, Bank.preset(gpu.PRESET_P25_C4FM, len(bins), 50000.0, fir, max_samples_per_call=n_ch))
        pipe.setChunks(8)
        return pipe

    want = build().process(x)
    pinned = C.c_void_p()
    gpu.check(L.sdrgpu_alloc_pinned(C.byref(pinned), x.nbytes))
    host = np.ctypeslib.as_array(C.cast(pinned, C.POINTER(C.c_float)), shape=(x.size,))
    stride = 4096
    d_sym, d_cnt = C.c_void_p(), C.c_void_p()
    gpu.check(L.sdrgpu_device_alloc(C.byref(d_sym), len(bins) * stride))
    gpu.check(L.sdrgpu_device_alloc(C.byref(d_cnt), 4 * len(bins)))
    for _ in range(3):
        pipe = build()
        host[:] = x
        gpu.check(L.sdrgpu_pipeline_process(pipe._h, pinned, x.size, gpu.HOST, d_sym, stride, None, 0, d_cnt, gpu.DEVICE))
        host[:] = 7.0                                         # the caller reuses its buffer right away
        pipe.bank.sync()
        sym = np.zeros((len(bins), stride), np.uint8)
        cnt = np.zeros(len(bins), np.int32)
        gpu.check(L.sdrgpu_memcpy(gpu.ptr(sym), d_sym, sym.nbytes, gpu.HOST, gpu.DEVICE))
        gpu.check(L.sdrgpu_memcpy(gpu.ptr(cnt), d_cnt, cnt.nbytes, gpu.HOST, gpu.DEVICE))
        for k in range(len(bins)):
            assert cnt[k] == want[k].size and np.array_equal(sym[k, :cnt[k]], want[k]), k
    L.sdrgpu_device_free(d_sym)
    L.sdrgpu_device_free(d_cnt)
    L.sdrgpu_free_pinned(pinned)


def test_config5_shape_800_channels_pipeline(gpu):
    """BASELINE configs[4], one tuner: 20 MS/s, M = 800, every bin carries C4FM, all 800 channels through the fused
    pipeline (pfb2_kernel<800, 32, 25> direct row stores -> FIR -> AGC -> demodulator).  Every channel must decode its
    transmitted dibits, and a sample of rows -- first / last, both sides of the 32 x 25 factorisation's row groups, the
    spectrum edge -- is bit-exact against the oracle chain fed the same channel I/Q, whose channel I/Q in turn is within
    1e-4 of the oracle channelizer's."""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 800, 4 * 1024
    rng = np.random.default_rng(46)
    dibs = [rng.integers(0, 4, int(n_ch * 0.096) + 8) for _ in range(m)]
    base = [sg.c4fm(dibs[k], carrier_offset=rng.uniform(-200, 200), timing_phase=rng.uniform(0, 1), n_samples=n_ch,
                    amplitude=0.01, phase0=rng.uniform(0, 6.28)) for k in range(m)]
    x = sg.interleave(sg.multiplex(base, list(range(m)), m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-3))
    fir = c4fm_taps()
    chan = ComplexPolyphaseChannelizerM2(2e7, 9, maxInputFloats=x.size)
    assert chan.getChannelCount(2e7) == 800
    pipe = Pipeline(chan, Bank.preset(gpu.PRESET_P25_C4FM, m, 50000.0, fir, max_samples_per_call=n_ch))
    got = pipe.process(x)
    assert len(got) == m
    scores = np.array([_score(got[k], dibs[k], skip=200) for k in range(m)])
    assert np.mean(scores > 0.95) > 0.9, np.sort(scores)[:10]   # (390 symbols per channel: some are still acquiring)
    slow = [int(k) for k in np.nonzero(scores <= 0.95)[0]][:8]
    iq = ComplexPolyphaseChannelizerM2(2e7, 9, maxInputFloats=x.size).receiveChannels(x)
    head = 512                                                  # blocks of the (slow) float64-DFT oracle channelizer
    res = oracle.Channelizer(oracle.sinc_m2_channelizer(25000.0, m, 9), m).receive(x[:2 * head * (m // 2)], mode="f64")
    for k in [0, 1, 24, 25, 31, 32, 399, 400, 401, 767, 768, 799] + slow:
        want = oracle.P25Chain(oracle.C4FM, 50000.0, fir).receive(iq[k])
        assert np.array_equal(got[k], want), k
        y = oracle.OneChannelOutputProcessor(50000.0, k, float(m)).process(res)
        assert sg.rel_rms(iq[k][:2 * head], y) < TOL, k


@pytest.mark.parametrize("world", [2, 3])
def test_level2_bin_slices_equal_the_unsharded_pipeline(gpu, world):
    """SURVEY.md 8e level 2 on the device: every "rank" channelizes the same tuner buffer and keeps its slice of the bins
    (sharding.bin_slice); the slices' dibits, put together, are those of the unsharded run -- all M = 96 bins busy."""
    from sdrtrunk_b200 import sharding
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 4 * 1024
    rng = np.random.default_rng(81)
    x = _tuner_stream(rng, m, n_ch, list(range(m)))
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()

    def run(lo, hi):
        chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
        if (lo, hi) != (0, m):
            chan.setChannels(list(range(lo, hi)))
        return Pipeline(chan, Bank.preset(gpu.PRESET_P25_C4FM, hi - lo, 50000.0, fir, max_samples_per_call=n_ch)).process(x)

    want = run(0, m)
    got = []
    for rank in range(world):
        got += run(*sharding.bin_slice(m, rank, world))
    assert len(got) == m
    for k in range(m):
        assert np.array_equal(got[k], want[k]), k
