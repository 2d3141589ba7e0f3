"""sdrgpu_chan_set_frequency_offsets against the oracle's stateful output processors.

The reference changes a running channel's offset with ChannelOutputProcessor.setFrequencyOffset between two
processChannelResults calls: only the Oscillator's angle changes, the phasor carries on, a one-bin channel stops mixing at
offset 0 (holding its phasor) and resumes from it later; two-bin channels keep their synthesizer.  Each case keeps one
oracle One/TwoChannelOutputProcessor per channel for the whole stream, fed the device's own results layout call by call,
and calls set_frequency_offset at the same call boundaries as the channelizer.  Every row must be bit-exact, and the
rows of channels not yet changed must equal a run without changes.  The calls are ragged (some complete no block) and
the look-ahead rings are small, so changes land across ring wraps, right after a selection (nothing produced ahead) and
after a switch from no mixed channel at all (a call longer than the look-ahead).  Pipelines: a change lands with one
call (single pass) or two calls (filters-first, submit / wait) produced ahead, and routed rows follow the channelizer.
"""
import ctypes as C

import numpy as np
import pytest

import oracle
from test_bank_gpu import _tuner_stream, c4fm_taps
from test_channelizer_paths_gpu import CH_RATE, _input, _selection, _synth, _taps

MAX_BLOCKS = 64      # blocks per call the channelizers are sized for: rings of 2 x 64 + 9 slots wrap every few calls


def _calls(m, rng, n_calls=44):
    """ragged call sizes in complex samples: empty calls, calls that complete no block, whole look-aheads"""
    sizes = []
    for i in range(n_calls):
        kind = i % 6
        if kind == 0:
            sizes.append(int(rng.integers(0, m // 2)))                      # at most one block
        elif kind == 3:
            sizes.append(MAX_BLOCKS * (m // 2) - int(rng.integers(0, m // 2)))   # a full call
        else:
            sizes.append(int(rng.integers(1, MAX_BLOCKS)) * (m // 2) + int(rng.integers(0, m // 2)))
    return sizes


def _schedule(entries, n_calls, rng, start_plain):
    """{call: {channel: offset}}: nonzero -> nonzero, -> 0, back to nonzero (the held phasor), 0 -> nonzero of plain
    channels, every channel at once, repeats of the current value; entries[i][1] is the starting offset"""
    n = len(entries)
    cur = [off for _, off, _ in entries]
    one = [i for i in range(n) if len(entries[i][0]) == 1]
    new = lambda: int(rng.integers(1, 12000)) * int(rng.choice([-1, 1]))
    plan = {}

    def change(call, chans, value=None):
        step = plan.setdefault(call, {})
        for i in chans:
            step[i] = new() if value is None else value
            cur[i] = step[i]

    pick = lambda pool, k: [int(i) for i in rng.choice(pool, min(k, len(pool)), replace=False)] if pool else []
    nz = lambda: [i for i in range(n) if cur[i] != 0]
    if not start_plain:
        change(0, pick(nz(), n // 3))                                   # before any block: nothing produced ahead
    change(2, pick(nz(), n // 4))                                       # nonzero -> nonzero (two-bin channels too)
    stopped = pick([i for i in nz() if i in one], max(2, n // 6))
    change(5, stopped, 0)                                               # -> 0: hold the phasor
    change(6, pick(nz(), 3))
    change(9, stopped)                                                  # back to nonzero: resume from it
    change(9, pick([i for i in one if cur[i] == 0], max(2, n // 8)))    # plain -> corrected
    change(13, pick(nz(), 5))
    change(14, stopped[:1], 0)
    plan.setdefault(17, {}).update({i: cur[i] for i in pick(list(range(n)), n // 3)})   # repeats of the same value
    change(18, stopped[:1])
    change(22, list(range(n)))                                          # every channel at once (plain -> fused path)
    change(27, pick(one, n // 5), 0)
    change(31, [i for i in one if cur[i] == 0][:max(1, n // 10)])
    change(35, pick(nz(), n // 2))
    assert max(plan) < n_calls
    return plan


def _processors(entries):
    procs = []
    for idx, off, g in entries:
        p = (oracle.TwoChannelOutputProcessor(CH_RATE, idx[0], idx[1], _synth(), g) if len(idx) == 2 else
             oracle.OneChannelOutputProcessor(CH_RATE, idx[0], g))
        p.set_frequency_offset(off)
        procs.append(p)
    return procs


def _chan(m, fmt, entries):
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    ch = ComplexPolyphaseChannelizerM2(_taps(m, 9), 25000 * m, m, maxInputFloats=2 * MAX_BLOCKS * (m // 2))
    if fmt != "f32":
        ch.setSampleFormat(fmt)
    if entries is not None:
        ch.setOutputChannels(entries, _synth())
    return ch


# every bin corrected at gain M (pfb2_kernel's fused mix at M = 400 / 800), the paths test's mixed selection D (two-bin,
# corrected and plain one-bin channels, double gains), and every bin plain until the changes make them corrected
KINDS = ["Cf", "D", "plain"]
CASES = [pytest.param(m, fmt, k, id="%d-%s-%s" % (m, fmt, k))
         for m, fmt in ((96, "f32"), (400, "f32"), (400, "u8"), (800, "f32"), (800, "u8")) for k in KINDS]


@pytest.mark.gpu
@pytest.mark.parametrize("m, fmt, kind", CASES)
def test_channel_rows_follow_the_oracle_through_offset_changes(gpu, m, fmt, kind):
    rng = np.random.default_rng(m + len(kind) + len(fmt))
    entries = [([b], 0, float(m)) for b in range(m)] if kind == "plain" else _selection(kind, m)
    raw, _ = _input(m, fmt)
    sizes = _calls(m, rng)
    per = 2   # raw values per complex sample: I and Q
    need = per * sum(sizes)
    reps = -(-need // raw.size)
    raw = np.concatenate([raw] * reps)[:need]
    plan = _schedule(entries, len(sizes), rng, kind == "plain")

    res_chan, ch, still = _chan(m, fmt, None), _chan(m, fmt, entries), _chan(m, fmt, entries)
    procs = _processors(entries)
    changed = set()
    pos = 0
    for ci, n in enumerate(sizes):
        part = raw[pos:pos + per * n]
        pos += per * n
        if ci in plan:
            ch.setFrequencyOffsets(plan[ci])
            for i, off in plan[ci].items():
                procs[i].set_frequency_offset(off)
                if off != entries[i][1] or i in changed:
                    changed.add(i)
        res = res_chan.receive(part)
        got = ch.receiveChannels(part)
        base = still.receiveChannels(part)
        assert got.shape == (len(entries), 2 * res.shape[0])
        want = [p.process(res) for p in procs]
        bad = [i for i in range(len(entries)) if not np.array_equal(got[i], want[i])]
        assert not bad, (ci, [(i, entries[i][0]) for i in bad[:4]])
        same = [i for i in range(len(entries)) if i not in changed]
        assert np.array_equal(got[same], base[same]), ci


@pytest.mark.gpu
def test_routed_pipeline_returns_the_changed_rows(gpu):
    """a pipeline splitting the mixed selection over two pass-through banks (the ROUTED kernel instances) returns, after
    every change, the rows a channelizer alone returns, bit for bit"""
    from sdrtrunk_b200.dsp import Bank, Pipeline
    m, fmt = 400, "f32"
    rng = np.random.default_rng(11)
    entries = _selection("D", m)
    n_rows = len(entries)
    raw, _ = _input(m, fmt)
    sizes = [48 * (m // 2)] * 6
    plan = _schedule(entries, 40, rng, False)
    plan = {k: plan[k] for k in sorted(plan)[:6]}
    steps = dict(zip(range(6), plan.values()))
    route = [int(r) for r in rng.integers(0, 2, n_rows)]
    route[:2] = [0, 1]
    banks = [Bank(route.count(j), CH_RATE, block_size=16, max_samples_per_call=2 * MAX_BLOCKS) for j in range(2)]
    routed_chan, alone = _chan(m, fmt, entries), _chan(m, fmt, entries)
    pipe = Pipeline(routed_chan, banks=banks, route=route)
    pos = 0
    for ci, n in enumerate(sizes):
        part = raw[2 * pos:2 * (pos + n)]
        pos += n
        if ci in steps:
            routed_chan.setFrequencyOffsets(steps[ci])
            alone.setFrequencyOffsets(steps[ci])
        out = pipe.process(part)
        want = alone.receiveChannels(part)
        rows = np.empty_like(want)
        for j in range(2):
            rows[[i for i in range(n_rows) if route[i] == j]] = out[j]
        assert np.array_equal(rows, want), ci
    pipe.dispose()


@pytest.mark.gpu
def test_offset_changes_through_the_pipeline_schedules(gpu):
    """Two tuners feed a C4FM bank; offsets change between calls (nonzero -> nonzero, -> 0, back, every channel).  The
    dibits are identical through the single pass (one call produced ahead), the filters-first schedule on device input
    (two calls ahead, producer at the start of the call), submit / wait with the change issued while two calls are in
    flight (applied from the next submit), and the reference sequence receiveChannels -> Bank.process."""
    from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
    m, n_ch = 96, 30 * 1024
    rng = np.random.default_rng(97)
    bins = [[2, 30, 77], [5, 6, 95]]
    offsets = [[37, -53, 120], [-200, 9, 0]]
    xs = [_tuner_stream(rng, m, n_ch, b) for b in bins]
    taps, fir = oracle.sinc_m2_channelizer(25000.0, m, 9), c4fm_taps()
    rows = sum(len(b) for b in bins)
    unit = m * 1024
    sizes = [6 * unit, 8 * unit, 3 * unit, 8 * unit, 5 * unit]
    sizes.append(xs[0].size - sum(sizes))
    edges = np.cumsum([0] + sizes)
    # per call: {tuner: {channel: offset}}
    plan = {1: {0: {1: -310}, 1: {2: 75}},
            2: {0: {0: 0, 2: 400}, 1: {0: -150}},
            3: {1: {1: 0}},
            4: {0: {0: 61, 1: -80, 2: 0}, 1: {0: 33, 1: 250, 2: 0}},
            5: {0: {0: 61, 2: -12}, 1: {1: -250}}}

    def chans():
        out = []
        for k in range(2):
            ch = ComplexPolyphaseChannelizerM2(taps, 2400000, m, maxInputFloats=8 * unit)
            ch.setOutputChannels([([b], off) for b, off in zip(bins[k], offsets[k])])
            out.append(ch)
        return out

    def pipeline(device_chunks):
        cs = chans()
        pipe = Pipeline(cs, Bank.preset(gpu.PRESET_P25_C4FM, rows, 50000.0, fir, max_samples_per_call=9 * 1024))
        pipe.setChunks(1)
        pipe.setDeviceChunks(device_chunks)
        return pipe, cs

    def apply(cs, i):
        for k, step in plan.get(i, {}).items():
            cs[k].setFrequencyOffsets(step)

    single, cs = pipeline(1)
    want = []
    for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
        apply(cs, i)
        want.append(single.process([x[a:b] for x in xs]))
    assert sum(w.size for w in want[2]) > 1000

    # the reference sequence: the channelizers' rows through a bank of their own
    cs = chans()
    bank = Bank.preset(gpu.PRESET_P25_C4FM, rows, 50000.0, fir, max_samples_per_call=9 * 1024)
    for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
        apply(cs, i)
        got = bank.process(np.concatenate([c.receiveChannels(x[a:b]) for c, x in zip(cs, xs)]))
        for r in range(rows):
            assert np.array_equal(got[r], want[i][r]), ("reference", i, r)

    first, cs = pipeline(2)   # device-resident input, two time chunks: the filters-first schedule
    L = gpu.lib()
    for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
        apply(cs, i)
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

    stream, cs = pipeline(2)
    got = []
    for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
        stream.submit([x[a:b].copy() for x in xs])
        apply(cs, i + 1)          # calls i - 1 and i in flight: applies from submit i + 1
        if i >= 1:
            got.append(stream.wait())
    got.append(stream.wait())
    for i in range(len(want)):
        for r in range(rows):
            assert np.array_equal(got[i][r], want[i][r]), ("stream", i, r)
