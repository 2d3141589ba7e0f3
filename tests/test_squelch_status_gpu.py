"""Squelch status per assembler buffer (sdrgpu_bank_set_squelch_reporting) and per-channel squelch thresholds
(sdrgpu_bank_set_squelch_threshold) of SquelchingFMDemodulator banks, on both FM paths (nbfm_fused_kernel and the
five-kernel path), through banks, pipelines and routed pipelines.  The reference side is the oracle's
SquelchingFMDemodulator driven buffer by buffer: the expected byte after each buffer is state | squelch_changed << 2."""
import ctypes as C

import numpy as np
import pytest

import oracle
import siggen as sg

pytestmark = pytest.mark.gpu


def _oracle_fm(bufs, alpha, threshold_db, ramp, thresholds_at=None):
    """oracle SquelchingFMDemodulator over a list of buffers (already filtered): (audio, status bytes).
    thresholds_at: {buffer index: dB} threshold changes applied before that buffer."""
    fm = oracle.SquelchingFMDemodulator(alpha, threshold_db, ramp)
    audio, status = [], []
    for i, buf in enumerate(bufs):
        if thresholds_at and i in thresholds_at:
            fm.s.sq.threshold = 10.0 ** (thresholds_at[i] / 10.0)
        audio.append(fm.demodulate(buf))
        status.append(fm.s.sq.state | fm.s.squelch_changed << 2)
    return np.concatenate(audio), np.array(status, np.uint8)


def _front_end(x, block, rate, fir, agc=False):
    """the oracle's decimator -> ComplexFIR [-> AGC] of one channel, buffer by buffer"""
    dec = oracle.Decimator(rate) if rate else None
    f = oracle.ComplexFIR(fir) if fir is not None else None
    out = []
    for b in range(x.size // (2 * block)):
        y = x[2 * block * b:2 * block * (b + 1)]
        y = dec.decimate_complex(y) if dec else y
        y = f.filter(y) if f is not None else y
        out.append(oracle.agc_block(y) if agc else y)
    return out


def _nbfm_channels(rng, c, n, fs, quiet):
    x = []
    for k in range(c):
        loud = sg.nbfm(fs, n, audio_hz=300.0 * (k + 1), carrier_offset=150.0 * k, amplitude=0.3) + sg.awgn(rng, n, 1e-3)
        env = np.ones(n)
        q0 = (k * 997) % (n // 2)
        env[q0:q0 + n // 4] = quiet                    # a quiet stretch somewhere: the squelch closes
        x.append(sg.interleave(loud * env))
    return np.stack(x)


def _run(bank, x, cuts, block, want_squelch=True):
    outs = [bank.process(x[:, 2 * a * block:2 * b * block], want_squelch=want_squelch) for a, b in zip(cuts[:-1], cuts[1:])]
    if not want_squelch:
        return np.concatenate(outs, axis=1)
    return np.concatenate([o[0] for o in outs], axis=1), np.concatenate([o[1] for o in outs], axis=1)


@pytest.mark.parametrize("ramp", [4, 0])
@pytest.mark.parametrize("rate", [0, 2, 4, 8])
def test_fused_kernel_statuses(gpu, rate, ramp):
    """nbfm_fused_kernel, decimation 0 / 2 / 4 / 8 (outputs per buffer 1024 .. 128 against 256-output tiles), 7 channels,
    calls of 3, 1, 5 and 2 buffers: statuses equal the oracle byte for byte, and the audio with reporting on is
    bit-identical to the audio of a bank without it"""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(140 + rate)
    d, c, block = max(rate, 1), 7, 1024
    n = 11 * block
    fir = oracle.nbfm_iq_taps() if rate != 4 else oracle.nbfm_iq_taps()[4:-4]
    x = _nbfm_channels(rng, c, n, 25000.0 * d, 1e-5)
    kw = dict(demod=gpu.DEMOD_FM_SQUELCH, fir_taps=fir, decimation=rate, squelch_alpha=0.01, squelch_threshold_db=-40.0,
              squelch_ramp=ramp, block_size=block, max_samples_per_call=8 * block)
    cuts = [0, 3, 4, 9, 11]
    audio, status = _run(Bank(c, 25000.0 * d, **kw), x, cuts, block)
    plain = _run(Bank(c, 25000.0 * d, **kw), x, cuts, block, want_squelch=False)
    assert status.shape == (c, 11)
    assert np.array_equal(audio.view(np.uint32), plain.view(np.uint32))
    for k in range(c):
        want_audio, want = _oracle_fm(_front_end(x[k], block, rate, fir), 0.01, -40.0, ramp)
        assert np.array_equal(audio[k] == 0.0, want_audio == 0.0), k
        assert np.array_equal(status[k], want), (k, status[k], want)
        assert np.any(want & gpu.SQUELCH_CHANGED) and np.any(want == gpu.SQUELCH_UNMUTE), k


@pytest.mark.parametrize("rate, agc", [(16, False), (32, False), (4, True)])
def test_five_kernel_path_statuses(gpu, rate, agc):
    """squelch_gate_kernel (four half-band stages, an 11-tap first stage, block AGC): the same comparison"""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(160 + rate)
    c, block = 3, 2048
    n = 4096 * rate
    fir = oracle.nbfm_iq_taps()
    x = []
    for k in range(c):
        loud = sg.nbfm(25000.0 * rate, n, audio_hz=300.0 * (k + 1), carrier_offset=150.0 * k, amplitude=0.3) + sg.awgn(rng, n, 1e-3)
        env = np.ones(n)
        q0 = n // 8 + k * n // 16
        env[q0:q0 + 3 * n // 8] = 1e-7
        x.append(sg.interleave(loud * env))
    x = np.stack(x)
    kw = dict(demod=gpu.DEMOD_FM_SQUELCH, fir_taps=fir, decimation=rate, agc=agc, squelch_alpha=0.01,
              squelch_threshold_db=-40.0, squelch_ramp=4, block_size=block, max_samples_per_call=n // 2)
    cuts = sorted({0, 3, 4, n // block // 2, n // block})
    audio, status = _run(Bank(c, 25000.0 * rate, **kw), x, cuts, block)
    plain = _run(Bank(c, 25000.0 * rate, **kw), x, cuts, block, want_squelch=False)
    assert np.array_equal(audio.view(np.uint32), plain.view(np.uint32))
    for k in range(c):
        _, want = _oracle_fm(_front_end(x[k], block, rate, fir, agc), 0.01, -40.0, 4)
        assert np.array_equal(status[k], want), (k, status[k], want)
        assert np.sum((want & gpu.SQUELCH_CHANGED) != 0) >= 2, k


@pytest.mark.parametrize("agc", [False, True])
@pytest.mark.parametrize("ramp", [0, 4])
def test_status_edge_cases(gpu, ramp, agc):
    """alpha = 1 and no filters: the squelch compares each sample's own power, so edges can be placed exactly.
    Channel 0 opens and closes inside one buffer; channel 1 changes state on the first sample of buffers 3 and 5;
    channel 2's calls end while the ramp is in ATTACK and in DECAY (ramp 4); channel 3 is loud throughout.  agc: the
    five-kernel path (exact zeros stay zero behind the block AGC), else nbfm_fused_kernel."""
    from sdrtrunk_b200.dsp import Bank
    c, block, n_buf = 4, 256, 9
    n = n_buf * block
    z = np.zeros((c, n), np.complex128)
    loud = sg.tone(25000.0, 1000.0, n, 0.5)
    z[0, 2 * block + 50:2 * block + 120] = loud[2 * block + 50:2 * block + 120]
    z[1, 3 * block - ramp:5 * block - ramp] = loud[3 * block - ramp:5 * block - ramp]
    z[2, 4 * block - 2:7 * block - 2] = loud[4 * block - 2:7 * block - 2]
    z[3] = loud
    x = np.stack([sg.interleave(r) for r in z])
    cuts = [0, 2, 4, 7, 9]
    bank = Bank(c, 25000.0, demod=gpu.DEMOD_FM_SQUELCH, agc=agc, squelch_alpha=1.0, squelch_threshold_db=-20.0,
                squelch_ramp=ramp, block_size=block, max_samples_per_call=4 * block)
    _, status = _run(bank, x, cuts, block)
    want = [_oracle_fm(_front_end(x[k], block, 0, None, agc), 1.0, -20.0, ramp)[1] for k in range(c)]
    for k in range(c):
        assert np.array_equal(status[k], want[k]), (k, status[k], want[k])
    mute, unmute, changed = gpu.SQUELCH_MUTE, gpu.SQUELCH_UNMUTE, gpu.SQUELCH_CHANGED
    assert want[0][2] == mute | changed and want[0][1] == mute          # open and shut inside buffer 2
    before_open, before_shut = (gpu.SQUELCH_ATTACK, gpu.SQUELCH_DECAY) if ramp else (mute, unmute)
    assert want[1][3] == unmute | changed and want[1][2] == before_open   # the change is on buffer 3's first sample
    assert want[1][5] == mute | changed and want[1][4] == before_shut     # ... and on buffer 5's
    if ramp:
        assert want[2][3] == gpu.SQUELCH_ATTACK and want[2][6] == gpu.SQUELCH_DECAY   # calls end at buffers 4 and 7


@pytest.mark.parametrize("rate, agc", [(2, False), (16, False)])
def test_per_channel_thresholds(gpu, rate, agc):
    """every channel its own threshold; between calls a subset changes, then channel -1 sets all: equal to oracle
    instances whose threshold is set at the same buffer boundary, on both FM paths"""
    from sdrtrunk_b200.dsp import Bank
    rng = np.random.default_rng(180 + rate)
    c, block = 7, 1024
    n = 12 * block
    fir = oracle.nbfm_iq_taps()
    x = []
    for k in range(c):
        sig = sg.nbfm(25000.0 * rate, n, audio_hz=250.0 * (k + 1), amplitude=0.3) + sg.awgn(rng, n, 1e-3)
        env = np.repeat(10.0 ** (-rng.uniform(0.0, 3.0, n // 512) / 2.0), 512)    # levels 0 .. -60 dB
        x.append(sg.interleave(sig * env))
    x = np.stack(x)
    bank = Bank(c, 25000.0 * rate, demod=gpu.DEMOD_FM_SQUELCH, fir_taps=fir, decimation=rate, agc=agc, squelch_alpha=0.01,
                squelch_threshold_db=-40.0, squelch_ramp=4, block_size=block, max_samples_per_call=4 * block)
    first = [-15.0 - 7.0 * k for k in range(c)]
    plan = {0: {k: first[k] for k in range(c)}, 4: {1: -22.0, 4: -50.0, 6: -12.0}, 8: {-1: -30.0}}
    cuts = [0, 4, 8, 12]
    statuses = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        for ch, db in plan[a].items():
            bank.setSquelchThreshold(db, ch)
        statuses.append(bank.process(x[:, 2 * a * block:2 * b * block], want_squelch=True)[1])
    status = np.concatenate(statuses, axis=1)
    n_buf = n // block
    for k in range(c):
        at = {0: first[k]}
        if k in plan[4]:
            at[4] = plan[4][k]
        at[8] = plan[8][-1]
        _, want = _oracle_fm(_front_end(x[k], block, rate, fir, agc), 0.01, -40.0, 4, at)
        assert want.size == n_buf and np.array_equal(status[k], want), (k, status[k], want)
    assert len({tuple(s) for s in status}) > 2    # the thresholds make a difference


def _m96_nbfm_stream(rng, m, n_ch, bins):
    """NBFM channels at 50 kHz on channelizer bins, each loud, then silent for half the stream, then loud again"""
    base = []
    for i, _ in enumerate(bins):
        sig = sg.nbfm(50000.0, n_ch, audio_hz=400.0 * (i + 1), carrier_offset=100.0 * i, amplitude=0.3)
        env = np.ones(n_ch)
        q0 = n_ch // 8 + (i * 3331) % (n_ch // 8)
        env[q0:q0 + n_ch // 2] = 0.0
        base.append(sig * env)
    return sg.interleave(sg.multiplex(base, bins, m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-6))


def _threshold_db(iq):
    """5 dB below the loud channels' power: with the preset's alpha (0.0004) the squelch closes within the silent
    halves (the preset's -78 dB would take seconds) and opens again behind them"""
    p = np.abs(sg.deinterleave(np.concatenate(list(iq)))) ** 2
    return float(10.0 * np.log10(np.percentile(p, 90)) - 5.0)


def _oracle_from_channels(iq, fir, n_buf, threshold_db):
    """statuses of the NBFM preset (decimation 2, alpha 0.0004, ramp 4) over the GPU channelizer's output"""
    out = []
    for row in iq:
        row = row[:n_buf * 2 * 1024]
        out.append(_oracle_fm(_front_end(row, 1024, 2, fir), 0.0004, -78.0, 4, {0: threshold_db})[1])
    return np.stack(out)


def test_pipeline_statuses_host_and_device_outputs(gpu):
    """the configs[0] chain (2.4 MS/s, M = 96, 50 kHz channels, NBFM preset) through sdrgpu_pipeline_process: host and
    device outputs, chunks 1 and 8, calls that end inside a buffer -- the same statuses, equal to the oracle fed the
    channelizer's output"""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch, bins = 96, 16 * 1024, [4, 20, 33]
    rng = np.random.default_rng(7)
    x = _m96_nbfm_stream(rng, m, n_ch, bins)
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), oracle.nbfm_iq_taps()
    cut = x.size // 3 // 2 * 2
    L = gpu.lib()
    chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
    chan.setChannels(bins)
    iq = chan.receiveChannels(x)
    thr = _threshold_db(iq)

    def pipeline(chunks):
        chan = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
        chan.setChannels(bins)
        bank = Bank.preset(gpu.PRESET_NBFM, len(bins), 50000.0, fir, max_samples_per_call=n_ch)
        bank.setSquelchThreshold(thr)
        pipe = Pipeline(chan, bank)
        pipe.setChunks(chunks)
        return pipe, bank

    results = {}
    for chunks in (1, 8):
        pipe, _ = pipeline(chunks)
        parts = [pipe.process(x[:cut], want_squelch=True), pipe.process(x[cut:], want_squelch=True)]
        results[("host", chunks)] = (np.concatenate([p[0] for p in parts], axis=1), np.concatenate([p[1] for p in parts], axis=1))
        pipe, bank = pipeline(chunks)
        gpu.check(L.sdrgpu_bank_set_squelch_reporting(bank._h, 1))
        c, stride, dstride = len(bins), 24, n_ch
        d_sym, d_dem, d_cnt = C.c_void_p(), C.c_void_p(), C.c_void_p()
        gpu.check(L.sdrgpu_device_alloc(C.byref(d_sym), c * stride))
        gpu.check(L.sdrgpu_device_alloc(C.byref(d_dem), 4 * c * dstride))
        gpu.check(L.sdrgpu_device_alloc(C.byref(d_cnt), 4 * c))
        dem_parts, st_parts = [], []
        for seg in (x[:cut], x[cut:]):
            seg = np.ascontiguousarray(seg)
            gpu.check(L.sdrgpu_pipeline_process(pipe._h, gpu.ptr(seg), seg.size, gpu.HOST, d_sym, stride, d_dem, dstride,
                                                d_cnt, gpu.DEVICE))
            bank.sync()
            sym = np.zeros((c, stride), np.uint8)
            dem = np.zeros((c, dstride), np.float32)
            cnt = np.zeros(c, np.int32)
            gpu.check(L.sdrgpu_memcpy(gpu.ptr(sym), d_sym, sym.nbytes, gpu.HOST, gpu.DEVICE))
            gpu.check(L.sdrgpu_memcpy(gpu.ptr(dem), d_dem, dem.nbytes, gpu.HOST, gpu.DEVICE))
            gpu.check(L.sdrgpu_memcpy(gpu.ptr(cnt), d_cnt, cnt.nbytes, gpu.HOST, gpu.DEVICE))
            nb = int(cnt[0]) // 512
            dem_parts.append(dem[:, :cnt[0]])
            st_parts.append(sym[:, :nb])
        for d in (d_sym, d_dem, d_cnt):
            L.sdrgpu_device_free(d)
        results[("device", chunks)] = (np.concatenate(dem_parts, axis=1), np.concatenate(st_parts, axis=1))
    ref_audio, ref_status = results[("host", 1)]
    n_buf = ref_status.shape[1]
    assert n_buf == n_ch // 1024
    for key, (audio, status) in results.items():
        assert np.array_equal(status, ref_status), key
        assert np.array_equal(audio.view(np.uint32), ref_audio.view(np.uint32)), key
    want = _oracle_from_channels(iq, fir, n_buf, thr)
    assert np.array_equal(ref_status, want), (ref_status, want)
    assert np.all(np.sum((want & gpu.SQUELCH_CHANGED) != 0, axis=1) >= 2)


def test_routed_pipeline_statuses(gpu):
    """a routed pipeline of a C4FM bank and an NBFM bank with reporting on: the NBFM bank's audio and statuses equal
    those of its own one-bank pipeline and the oracle's, and the C4FM dibits those of a C4FM-only pipeline"""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 16 * 1024
    rng = np.random.default_rng(9)
    fm_bins, c4_bins = [4, 33], [12, 50, 70]
    x_fm = _m96_nbfm_stream(rng, m, n_ch, fm_bins)
    c4 = [sg.c4fm(rng.integers(0, 4, int(n_ch * 0.096) + 8), carrier_offset=100.0 * i, n_samples=n_ch, amplitude=0.05)
          for i in range(len(c4_bins))]
    x = (x_fm + sg.interleave(sg.multiplex(c4, c4_bins, m, n_ch))).astype(np.float32)
    taps, fir_fm, fir_c4 = oracle.sinc_m2_channelizer(25000.0, m, 9), oracle.nbfm_iq_taps(), oracle.c4fm_baseband_taps()
    sel = [4, 12, 50, 33, 70]
    route = [1, 0, 0, 1, 0]

    def chan_for(bins):
        ch = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=x.size)
        ch.setChannels(bins)
        return ch

    def c4_bank():
        return Bank.preset(gpu.PRESET_P25_C4FM, len(c4_bins), 50000.0, fir_c4, max_samples_per_call=n_ch)

    thr = _threshold_db(chan_for(fm_bins).receiveChannels(x))

    def fm_bank():
        b = Bank.preset(gpu.PRESET_NBFM, len(fm_bins), 50000.0, fir_fm, max_samples_per_call=n_ch)
        b.setSquelchThreshold(thr)
        return b

    cut = x.size // 3 // 2 * 2
    want_c4 = Pipeline(chan_for([12, 50, 70]), c4_bank())
    want_c4 = [np.concatenate(p) for p in zip(want_c4.process(x[:cut]), want_c4.process(x[cut:]))]
    one = Pipeline(chan_for(fm_bins), fm_bank())
    parts = [one.process(x[:cut], want_squelch=True), one.process(x[cut:], want_squelch=True)]
    want_audio = np.concatenate([p[0] for p in parts], axis=1)
    want_status = np.concatenate([p[1] for p in parts], axis=1)
    for chunks in (1, 8):
        pipe = Pipeline(chan_for(sel), banks=[c4_bank(), fm_bank()], route=route)
        pipe.setChunks(chunks)
        parts = [pipe.process(x[:cut], want_squelch=True), pipe.process(x[cut:], want_squelch=True)]
        dibits = [np.concatenate(p) for p in zip(parts[0][0], parts[1][0])]
        assert all(np.array_equal(a, b) for a, b in zip(dibits, want_c4)), chunks
        audio = np.concatenate([p[1][0] for p in parts], axis=1)
        status = np.concatenate([p[1][1] for p in parts], axis=1)
        assert np.array_equal(audio.view(np.uint32), want_audio.view(np.uint32)), chunks
        assert np.array_equal(status, want_status), chunks
    oracle_status = _oracle_from_channels(chan_for(fm_bins).receiveChannels(x), fir_fm, want_status.shape[1], thr)
    assert np.array_equal(want_status, oracle_status)
    assert np.all(np.sum((oracle_status & gpu.SQUELCH_CHANGED) != 0, axis=1) >= 2)


def test_reporting_off_leaves_symbols_untouched(gpu):
    """without reporting an FM bank ignores `symbols`, on the bank and through a pipeline; NULL symbols with reporting
    on writes nothing and changes nothing else"""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    rng = np.random.default_rng(3)
    c, block = 3, 1024
    x = _nbfm_channels(rng, c, 4 * block, 50000.0, 1e-5)
    L = gpu.lib()
    bank = Bank.preset(gpu.PRESET_NBFM, c, 50000.0, oracle.nbfm_iq_taps(), max_samples_per_call=4 * block)
    sym = np.full((c, 8), 0xAB, np.uint8)
    dem = np.zeros((c, 2 * block), np.float32)
    gpu.check(L.sdrgpu_bank_process(bank._h, gpu.ptr(x), x.shape[1], 4 * block, gpu.HOST, gpu.ptr(sym), 8, gpu.ptr(dem),
                                    dem.shape[1], None, gpu.HOST))
    assert np.all(sym == 0xAB)
    ref = Bank.preset(gpu.PRESET_NBFM, c, 50000.0, oracle.nbfm_iq_taps(), max_samples_per_call=4 * block)
    gpu.check(L.sdrgpu_bank_set_squelch_reporting(ref._h, 1))
    dem2 = np.zeros_like(dem)
    gpu.check(L.sdrgpu_bank_process(ref._h, gpu.ptr(x), x.shape[1], 4 * block, gpu.HOST, None, 0, gpu.ptr(dem2),
                                    dem2.shape[1], None, gpu.HOST))
    assert np.array_equal(dem.view(np.uint32), dem2.view(np.uint32))
    m, n_ch = 96, 4 * 1024
    xs = _m96_nbfm_stream(rng, m, n_ch, [4, 20])
    chan = ComplexPolyphaseChannelizerM2(oracle.sinc_m2_channelizer(25000.0, m, 9), 2400000, m, maxInputFloats=xs.size)
    chan.setChannels([4, 20])
    pipe = Pipeline(chan, Bank.preset(gpu.PRESET_NBFM, 2, 50000.0, oracle.nbfm_iq_taps(), max_samples_per_call=n_ch))
    sym = np.full((2, 8), 0xCD, np.uint8)
    dem = np.zeros((2, n_ch), np.float32)
    gpu.check(L.sdrgpu_pipeline_process(pipe._h, gpu.ptr(xs), xs.size, gpu.HOST, gpu.ptr(sym), 8, gpu.ptr(dem), n_ch, None,
                                        gpu.HOST))
    assert np.all(sym == 0xCD) and np.any(dem != 0.0)


def test_argument_checks_leave_the_bank_usable(gpu):
    """non-squelch banks, channels out of range, non-finite thresholds and a symbol_stride shorter than the call's
    buffers are refused with INVALID_ARG; the refused call consumes nothing and the bank carries on as if it had not
    been made"""
    from sdrtrunk_b200.dsp import Bank
    L = gpu.lib()
    invalid = gpu.ERR_INVALID_ARG
    for other in (Bank(2, 25000.0, demod=gpu.DEMOD_FM), Bank(2, 25000.0),
                  Bank.preset(gpu.PRESET_P25_C4FM, 2, 50000.0, oracle.c4fm_baseband_taps())):
        assert L.sdrgpu_bank_set_squelch_reporting(other._h, 1) == invalid
        assert L.sdrgpu_bank_set_squelch_threshold(other._h, 0, -40.0) == invalid
    rng = np.random.default_rng(5)
    c, block = 3, 1024
    x = _nbfm_channels(rng, c, 6 * block, 50000.0, 1e-5)
    bank, ref = (Bank.preset(gpu.PRESET_NBFM, c, 50000.0, oracle.nbfm_iq_taps(), max_samples_per_call=4 * block)
                 for _ in range(2))
    for ch, db in ((c, -40.0), (-2, -40.0), (0, float("nan")), (-1, float("inf")), (1, float("-inf"))):
        assert L.sdrgpu_bank_set_squelch_threshold(bank._h, ch, db) == invalid, (ch, db)
    assert b"finite" in L.sdrgpu_last_error() or b"range" in L.sdrgpu_last_error()
    gpu.check(L.sdrgpu_bank_set_squelch_reporting(bank._h, 1))
    first = np.ascontiguousarray(x[:, :2 * 3 * block])
    sym = np.full((c, 2), 0x5A, np.uint8)
    dem = np.zeros((c, 3 * 512), np.float32)
    assert L.sdrgpu_bank_process(bank._h, gpu.ptr(first), first.shape[1], 3 * block, gpu.HOST, gpu.ptr(sym), 2,
                                 gpu.ptr(dem), dem.shape[1], None, gpu.HOST) == invalid
    assert b"symbol_stride" in L.sdrgpu_last_error() and np.all(sym == 0x5A)
    got = _run(bank, x, [0, 3, 6], block)
    want = _run(ref, x, [0, 3, 6], block)
    assert np.array_equal(got[0].view(np.uint32), want[0].view(np.uint32)) and np.array_equal(got[1], want[1])


def test_host_mirror_follows_the_oracle(gpu):
    """SquelchingFMDemodulator.isSquelchChanged() / isMuted() after every buffer, with a threshold change midway"""
    from sdrtrunk_b200.dsp import SquelchingFMDemodulator
    rng = np.random.default_rng(11)
    block, n_buf = 1024, 16
    x = _nbfm_channels(rng, 1, n_buf * block, 25000.0, 1e-5)[0]
    dut = SquelchingFMDemodulator(0.01, -40.0, 4)
    ref = oracle.SquelchingFMDemodulator(0.01, -40.0, 4)
    assert not dut.isSquelchChanged() and dut.isMuted()
    seen = set()
    for b in range(n_buf):
        if b == 10:
            dut.setSquelchThreshold(-8.0)
            ref.s.sq.threshold = 10.0 ** (-8.0 / 10.0)
        buf = x[2 * block * b:2 * block * (b + 1)]
        got = dut.demodulate(buf)
        want = ref.demodulate(buf)
        assert np.array_equal(got == 0.0, want == 0.0), b
        assert dut.isSquelchChanged() == bool(ref.s.squelch_changed), b
        assert dut.isMuted() == (ref.s.sq.state in (gpu.SQUELCH_MUTE, gpu.SQUELCH_ATTACK)), b
        seen.add((dut.isSquelchChanged(), dut.isMuted()))
    assert len(seen) >= 3
