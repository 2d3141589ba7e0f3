"""sdrgpu_pipeline_create_routed / _process_routed: one channelizer pass feeding several banks (decoder types).  Every
bank's outputs must equal, bit for bit, those of a one-bank pipeline whose channelizers select only that bank's
channels, fed the same samples."""
import ctypes as C

import numpy as np
import pytest

import oracle
import siggen as sg

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _tuner_stream(rng, m, n_ch, bins):
    base = [sg.c4fm(rng.integers(0, 4, int(n_ch * 0.096) + 8), carrier_offset=rng.uniform(-200, 200),
                    timing_phase=rng.uniform(0, 1), n_samples=n_ch, amplitude=0.05) for _ in bins]
    return sg.interleave(sg.multiplex(base, bins, m, n_ch) + sg.awgn(rng, n_ch * m // 2, 1e-3))


def _banks(gpu, kinds, sizes, n_ch):
    """kinds: 'c4fm' (P25 phase 1 sync detector on), 'nbfm' (the fused NBFM kernel), 'none' (FIR only)"""
    from sdrtrunk_b200.dsp import Bank
    out = []
    for kind, n in zip(kinds, sizes):
        if kind == "c4fm":
            b = Bank.preset(gpu.PRESET_P25_C4FM, n, 50000.0, oracle.c4fm_baseband_taps(), max_samples_per_call=n_ch)
            b.setSyncDetector(gpu.SYNC_P25_PHASE1)
        elif kind == "nbfm":
            b = Bank.preset(gpu.PRESET_NBFM, n, 50000.0, oracle.nbfm_iq_taps(), max_samples_per_call=n_ch)
        else:
            b = Bank(n, 50000.0, fir_taps=oracle.c4fm_baseband_taps(), max_samples_per_call=n_ch)
        out.append(b)
    return out


def _feed(gpu, pipe, xs, device_input=False, cuts=()):
    """xs: one buffer per tuner, cut at `cuts`; returns the concatenated results of every call (a list per bank for a
    routed pipeline)"""
    edges = [0] + [c // 2 * 2 for c in cuts] + [xs[0].size]
    parts = []
    for a, b in zip(edges[:-1], edges[1:]):
        seg = [np.ascontiguousarray(x[a:b]) for x in xs]
        one = len(seg) == 1   # a one-tuner Pipeline takes its buffer, not a list
        if not device_input:
            parts.append(pipe.process(seg[0] if one else seg))
            continue
        L = gpu.lib()
        ptrs = []
        for s_ in seg:
            d = C.c_void_p()
            gpu.check(L.sdrgpu_device_alloc(C.byref(d), max(s_.nbytes, 16)))
            gpu.check(L.sdrgpu_memcpy(d, gpu.ptr(s_), s_.nbytes, gpu.DEVICE, gpu.HOST))
            ptrs.append(d)
        parts.append(pipe.process(ptrs[0].value if one else [d.value for d in ptrs], gpu.DEVICE, seg[0].size))
        for d in ptrs:
            L.sdrgpu_device_free(d)
    return parts


def _join(parts):
    """one bank's results over several calls: per-row dibit lists or [rows, n] float arrays"""
    if isinstance(parts[0], list):
        return [np.concatenate(p) for p in zip(*parts)]
    return np.concatenate(parts, axis=1)


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def _routed_equals_per_bank(gpu, m, xs, chan_for, sel, route, kinds, n_ch, schedules):
    """sel[k]: tuner k's output channels (setChannels bins or setOutputChannels entries); route[k][i]: the bank of its
    i-th channel.  Runs every schedule on a routed pipeline and compares with per-bank one-bank pipelines."""
    from sdrtrunk_b200.dsp import Pipeline
    n_banks = len(kinds)
    sizes = [sum(r.count(j) for r in route) for j in range(n_banks)]
    want = []
    for j in range(n_banks):
        chans = [chan_for(k, [s for s, r in zip(sel[k], route[k]) if r == j]) for k in range(len(xs))]
        pipe = Pipeline(chans, _banks(gpu, [kinds[j]], [sizes[j]], n_ch)[0])
        pipe.setChunks(1)
        want.append(_join(_feed(gpu, pipe, xs)))
    for kw in schedules:
        kw = dict(kw)
        chunks, device_chunks = kw.pop("chunks", 1), kw.pop("device_chunks", 1)
        pipe = Pipeline([chan_for(k, sel[k]) for k in range(len(xs))], banks=_banks(gpu, kinds, sizes, n_ch),
                        route=[r for rk in route for r in rk])
        pipe.setChunks(chunks)
        pipe.setDeviceChunks(device_chunks)
        parts = _feed(gpu, pipe, xs, **kw)
        for j in range(n_banks):
            got = _join([p[j] for p in parts])
            assert _same(got, want[j]), (kw, chunks, device_chunks, j)
    return want


SCHEDULES = (dict(chunks=8), dict(chunks=1), dict(chunks=3, cuts=(40000, 44000)),
             dict(device_input=True), dict(device_input=True, device_chunks=4))


@pytest.mark.parametrize("fmt", ["f32", "s8"])
def test_routed_pipeline_m96_three_decoders_equals_per_bank_pipelines(gpu, fmt):
    """three tuners at M = 96 (16-block tiles: the general store pass through the row table), their channels interleaved
    over a C4FM bank with the P25 phase 1 sync detector, an NBFM bank (fused kernel) and a DEMOD_NONE bank, under every
    schedule of the one-bank multi-tuner pipeline; one channel of each digital bank also against the oracle"""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m, n_ch = 96, 12 * 1024
    rng = np.random.default_rng(81)
    bins = [[2, 30, 77, 10], [5, 6, 60], [0, 47, 48, 95, 20]]
    route = [[0, 1, 2, 0], [1, 0, 2], [2, 0, 1, 0, 1]]
    xs = [_tuner_stream(rng, m, n_ch, b) for b in bins]
    if fmt == "s8":
        xs = [np.clip(np.round(x * 128.0 * 4), -128, 127).astype(np.int8) for x in xs]
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)

    def chan_for(k, sel):
        ch = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=xs[0].size)
        ch.setChannels(sel)
        ch.setSampleFormat(fmt)
        return ch

    want = _routed_equals_per_bank(gpu, m, xs, chan_for, bins, route, ["c4fm", "nbfm", "none"], n_ch, SCHEDULES)
    assert all(w.size > 1000 for w in want[0])
    if fmt == "f32":
        # tuner 1's bin 6 is the C4FM bank's row 2 (the dibit in the low bits of the sync detector's symbol bytes), its
        # bin 60 the DEMOD_NONE bank's row 1
        iq = chan_for(1, [6, 60]).receiveChannels(xs[1])
        fir = oracle.c4fm_baseband_taps()
        assert np.array_equal(want[0][2] & 3, oracle.P25Chain(oracle.C4FM, 50000.0, fir).receive(iq[0]))
        assert np.array_equal(want[2][1], oracle.ComplexFIR(fir).filter(iq[1]))


def test_routed_pipeline_m400_special_channels_and_fused_mix(gpu):
    """M = 400 (8-block tiles, direct row stores): two-bin and frequency-corrected channels routed to different banks
    (post_channel_kernel and osc_mix_kernel through the row table); then every bin frequency-corrected and split over two
    banks (the oscillator mix fused into pfb2_kernel's direct store)"""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m, n_ch = 400, 6 * 1024
    rng = np.random.default_rng(83)
    fs = 25000.0 * m
    xs = [_tuner_stream(rng, m, n_ch, b) for b in ([7, 20, 150], [3, 90, 300])]
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)

    def chan_for(k, sel):
        ch = ComplexPolyphaseChannelizerM2(taps, int(fs), m, maxInputFloats=xs[0].size)
        ch.setOutputChannels(sel)
        return ch

    sel = [[([7], 900), ([20, 21], -2500), ([150], 0), ([33], -1234, 2.5)],
           [([3], 0), ([90, 91], 0), ([300], 4000), ([301, 302], 1500)]]
    route = [[0, 1, 0, 1], [1, 0, 1, 0]]
    schedules = (dict(chunks=8), dict(chunks=1, cuts=(50000,)), dict(device_input=True, device_chunks=3))
    _routed_equals_per_bank(gpu, m, xs, chan_for, sel, route, ["c4fm", "none"], n_ch, schedules)

    offsets = [int(v) for v in rng.integers(-12000, 12000, m)]
    every = [[([b], offsets[b], float(m)) for b in range(m)]]
    split = [[int(v) for v in rng.integers(0, 2, m)]]
    _routed_equals_per_bank(gpu, m, xs[:1], chan_for, every, split, ["c4fm", "nbfm"], n_ch,
                            (dict(chunks=4), dict(device_input=True)))


def test_routed_pipeline_config5_shape(gpu):
    """one tuner at M = 800 (20 MS/s), all 800 bins split over a C4FM bank and an NBFM bank"""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m, n_ch = 800, 4 * 1024
    rng = np.random.default_rng(85)
    xs = [_tuner_stream(rng, m, n_ch, [1, 399, 400, 640, 799])]
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)

    def chan_for(k, sel):
        ch = ComplexPolyphaseChannelizerM2(taps, int(25000.0 * m), m, maxInputFloats=xs[0].size)
        ch.setChannels(sel)
        return ch

    route = [[1 if b % 5 == 4 else 0 for b in range(m)]]    # 640 C4FM, 160 NBFM
    _routed_equals_per_bank(gpu, m, xs, chan_for, [list(range(m))], route, ["c4fm", "nbfm"], n_ch,
                            (dict(chunks=8), dict(device_input=True)))


def test_routed_pipeline_argument_and_state_checks(gpu):
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 4 * 1024
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    chans = [ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=2 * 48 * n_ch) for _ in range(2)]
    for ch in chans:
        ch.setChannels([1, 2, 3])
    c4, fm = _banks(gpu, ["c4fm", "nbfm"], [4, 2], n_ch)
    L = native.lib()

    def create(banks, route, cs=chans):
        h = C.c_void_p()
        ch = (C.c_void_p * len(cs))(*[c._h if c is not None else None for c in cs])
        bk = (C.c_void_p * len(banks))(*[b._h if b is not None else None for b in banks])
        r = (C.c_int * len(route))(*route)
        st = L.sdrgpu_pipeline_create_routed(C.byref(h), ch, len(cs), bk, len(banks), r)
        if st == native.OK:
            L.sdrgpu_pipeline_destroy(h)
        return st

    ok = [0, 0, 1, 1, 0, 0]
    assert create([c4, fm], [0, 0, 2, 1, 0, 0]) == native.ERR_INVALID_ARG          # route entry out of range
    assert create([c4, fm], [0, -1, 1, 1, 0, 0]) == native.ERR_INVALID_ARG
    assert create([c4, c4], ok) == native.ERR_INVALID_ARG                          # the same bank twice
    assert create([c4, fm], [0, 0, 0, 1, 0, 0]) == native.ERR_INVALID_ARG          # 5 rows for a 4-channel bank
    assert create([c4, None], ok) == native.ERR_INVALID_ARG
    assert create([c4, fm], ok, [chans[0], None]) == native.ERR_INVALID_ARG
    other = ComplexPolyphaseChannelizerM2(oracle.sinc_m2_channelizer(25000.0, 160, 9), 4000000, 160)
    other.setChannels([1, 2, 3])
    assert create([c4, fm], ok, [chans[0], other]) == native.ERR_INVALID_ARG       # different channel counts
    odd = _banks(gpu, ["none"], [2], n_ch)[0]
    odd_block = type(odd)(2, 50000.0, block_size=512, max_samples_per_call=n_ch)
    assert create([c4, odd_block], ok) == native.ERR_INVALID_ARG                   # different block sizes
    odd.process(np.zeros((2, 2 * 100), np.float32))                                # 100 samples pending
    assert create([c4, odd], ok) == native.ERR_BAD_STATE
    assert create([c4, fm], ok) == native.OK                                       # ... and the handles still work

    pipe = Pipeline(chans, banks=[c4, fm], route=ok)
    xs = [_tuner_stream(np.random.default_rng(k), m, n_ch, [1, 2, 3]) for k in range(2)]
    ptrs = (C.c_void_p * 2)(*[x.ctypes.data for x in xs])
    sym = np.zeros((4, 64), np.uint8)
    assert L.sdrgpu_pipeline_process_multi(pipe._h, ptrs, xs[0].size, native.HOST, native.ptr(sym), 64, None, 0, None,
                                           native.HOST) == native.ERR_BAD_STATE
    assert L.sdrgpu_pipeline_submit_multi(pipe._h, ptrs, xs[0].size, native.ptr(sym), 64, None) == native.ERR_BAD_STATE
    assert L.sdrgpu_pipeline_process_routed(pipe._h, ptrs, xs[0].size, native.HOST, None, native.HOST) == native.ERR_INVALID_ARG
    got = pipe.process(xs)
    assert len(got) == 2 and len(got[0]) == 4 and got[1].shape[0] == 2
    chans[1].setChannels([1, 2])                                                   # the route was built for 3
    with pytest.raises(native.IllegalStateException):
        pipe.process(xs)
    pipe.dispose()
