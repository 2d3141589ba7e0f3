"""sdrgpu_chan_update_selection against the oracle's stateful output processors.

In the reference PolyphaseChannelManager adds and removes output processors, and moves one to other bins with
setPolyphaseChannelIndices; the other processors carry on untouched.  Each case keeps one oracle One/TwoChannel-
OutputProcessor per channel for the whole stream, fed the device's own results layout call by call: at an edit, kept
processors carry over (with a change of bins -- Moved below -- and set_frequency_offset where their entry changed) and
new entries get fresh ones.  Every row must be bit-exact, and the rows of channels kept unchanged since the start must equal
a run without edits.  The calls are ragged and the look-ahead rings small, so edits land across ring wraps, right after a
selection, and twice around a call that completes no block.
"""
import numpy as np
import pytest

import oracle
from test_bank_gpu import _tuner_stream, c4fm_taps
from test_channelizer_paths_gpu import CH_RATE, _input, _selection, _synth, _taps

MAX_BLOCKS = 64      # blocks per call the channelizers are sized for: rings of 2 x 64 + 9 slots wrap every few calls


def _calls(m, rng, n_calls=40):
    """ragged call sizes in complex samples; call 12 is empty (an edit on each side of it)"""
    sizes = []
    for i in range(n_calls):
        kind = i % 6
        if kind == 0:
            sizes.append(int(rng.integers(0, m // 2)))
        elif kind == 3:
            sizes.append(MAX_BLOCKS * (m // 2) - int(rng.integers(0, m // 2)))
        else:
            sizes.append(int(rng.integers(1, MAX_BLOCKS)) * (m // 2) + int(rng.integers(0, m // 2)))
    sizes[12] = 0
    return sizes


class Moved:
    """IPolyphaseChannelOutputProcessor.setPolyphaseChannelIndices (IPolyphaseChannelOutputProcessor.java:27-81, SURVEY
    section 8b) around an oracle processor: only the indexes change, the Oscillator, synthesizer and FS/4 position carry
    on.  The oracle processor keeps reading the bins it was created with, so it is fed results in which those columns
    hold the current bins.  Restated from the interface contract (the reference source is not available here): this
    behaviour is pinned only when the JVM harness runs (DESIGN section 8 item 8)."""

    def __init__(self, proc, idx):
        self.proc, self.created, self.idx = proc, list(idx), list(idx)

    def set_polyphase_channel_indices(self, idx):
        if len(idx) != len(self.created):
            raise ValueError("a processor keeps its bin count")
        self.idx = list(idx)

    def set_frequency_offset(self, offset):
        self.proc.set_frequency_offset(offset)

    def process(self, res):
        if self.idx != self.created:
            src = res
            res = res.copy()
            for a, b in zip(self.created, self.idx):
                res[:, 2 * a:2 * a + 2] = src[:, 2 * b:2 * b + 2]
        return self.proc.process(res)


class Entry:
    """one channel of the current selection: (indexes, offset, gain), the initial index it continues unchanged (or
    None once it was moved, retuned or restarted) and its oracle processor"""

    def __init__(self, idx, off, gain, origin=None, proc=None):
        self.idx, self.off, self.gain, self.origin = list(idx), int(off), float(gain), origin
        if proc is None:
            proc = (oracle.TwoChannelOutputProcessor(CH_RATE, idx[0], idx[1], _synth(), gain) if len(idx) == 2 else
                    oracle.OneChannelOutputProcessor(CH_RATE, idx[0], gain))
            proc.set_frequency_offset(off)
            proc = Moved(proc, idx)
        self.proc = proc

    def tuple(self):
        return (self.idx, self.off, self.gain)


def _edit(cur, spec):
    """spec: list of (previous index or -1, indexes, offset, gain) -> (new entries, previous list); kept processors
    follow the entry's new bins and offset"""
    new, prev = [], []
    for p, idx, off, gain in spec:
        if p < 0:
            new.append(Entry(idx, off, gain))
        else:
            e = cur[p]
            if list(idx) != e.idx:
                e.proc.set_polyphase_channel_indices(idx)
            if off != e.off:
                e.proc.set_frequency_offset(off)
            same = list(idx) == e.idx and off == e.off
            new.append(Entry(idx, off, gain, e.origin if same else None, e.proc))
        prev.append(p)
    return new, prev


def _keep(cur, i, idx=None, off=None):
    e = cur[i]
    return (i, e.idx if idx is None else idx, e.off if off is None else off, e.gain)


def _free_bins(cur, m, rng, k):
    """k first bins for channels, unused ones while there are enough (two channels may share a bin)"""
    used = {b for e in cur for b in e.idx}
    free = [b for b in range(m - 1) if b not in used]
    return [int(b) for b in rng.choice(free if len(free) >= k else range(m - 1), k, replace=False)]


def _plan(initial, m, rng):
    """{call: function(current entries) -> spec}: the edits of the issue, in an order that makes each reachable"""
    ones = lambda cur: [i for i, e in enumerate(cur) if len(e.idx) == 1]
    twos = lambda cur: [i for i, e in enumerate(cur) if len(e.idx) == 2]
    nz = lambda: int(rng.integers(1, 12000)) * int(rng.choice([-1, 1]))
    held = {}

    def restart_in_place(cur):              # before any block: nothing produced ahead
        return [(-1 if i % 7 == 3 else i,) + _keep(cur, i)[1:] for i in range(len(cur))]

    def remove_middle(cur):                 # later rows move up; leaves the fused / identity paths
        n = len(cur)
        gone = {n // 2 - 1, n // 2 + 1}
        return [_keep(cur, i) for i in range(n) if i not in gone]

    def append(cur):
        b = _free_bins(cur, m, rng, 3)
        return ([_keep(cur, i) for i in range(len(cur))] +
                [(-1, [b[0]], nz(), float(m)), (-1, [b[1]], 0, 2.5), (-1, [b[2], b[2] + 1], nz(), float(m))])

    def reverse(cur):
        return [_keep(cur, i) for i in reversed(range(len(cur)))]

    def retune(cur):                        # kept one-bin and two-bin channels to other bins, offsets of others
        spec = [_keep(cur, i) for i in range(len(cur))]
        one, two = ones(cur), twos(cur)
        b = _free_bins(cur, m, rng, 3)
        for k, i in enumerate(one[1:3]):
            spec[i] = _keep(cur, i, idx=[b[k]])
        if two:
            spec[two[0]] = _keep(cur, two[0], idx=[b[2], b[2] + 1])
        for i in one[4:4 + max(2, len(one) // 5)]:
            spec[i] = _keep(cur, i, off=nz())
        for i in two[1:2]:
            spec[i] = _keep(cur, i, off=nz())
        return spec

    def hold(cur):                          # a corrected one-bin channel goes to 0 (holds its phasor); order back
        spec = [_keep(cur, i) for i in reversed(range(len(cur)))]
        i = next(j for j in ones(cur) if cur[j].off != 0)
        held["proc"] = cur[i].proc
        spec[len(cur) - 1 - i] = _keep(cur, i, off=0)
        return spec

    def replace_class(cur):                 # class change by replacement: a new channel where a kept one was
        spec = [_keep(cur, i) for i in range(len(cur))]
        one = [i for i in ones(cur) if cur[i].proc is not held["proc"]]
        b = _free_bins(cur, m, rng, 1)
        spec[one[-1]] = (-1, [b[0], b[0] + 1], nz(), float(m))
        if twos(cur):
            spec[twos(cur)[0]] = (-1, [cur[twos(cur)[0]].idx[0]], nz(), 1.0 / 3)
        return spec

    def resume_moved(cur):                  # the held channel moves and resumes from its phasor
        spec = [_keep(cur, i) for i in range(len(cur))]
        i = next(j for j, e in enumerate(cur) if e.proc is held["proc"])
        spec[i] = _keep(cur, i, idx=_free_bins(cur, m, rng, 1), off=nz())
        return spec

    def restore(cur):                       # back to the initial selection: re-enters the fused / identity paths
        spec, taken = [], set()
        for idx, off, g in initial:
            hit = [i for i, e in enumerate(cur) if e.idx == list(idx) and e.gain == g and i not in taken]
            if hit:
                taken.add(hit[0])
                spec.append((hit[0], list(idx), off, g))
            else:
                spec.append((-1, list(idx), off, g))
        return spec

    def shuffle_with_offsets(cur):          # an arbitrary order and offset changes of kept entries at once
        order = [int(i) for i in rng.permutation(len(cur))]
        spec = [_keep(cur, i) for i in order]
        for k in range(0, len(spec), 3):
            i = spec[k][0]
            spec[k] = _keep(cur, i, off=0 if (len(cur[i].idx) == 1 and k % 2) else nz())
        return spec

    def drop_half(cur):
        return [_keep(cur, i) for i in range(0, len(cur), 2)]

    return {0: restart_in_place, 2: remove_middle, 4: append, 6: reverse, 8: retune, 10: hold, 12: replace_class,
            13: resume_moved, 16: restore, 20: shuffle_with_offsets, 24: restore, 28: drop_half, 31: append, 34: restore}


def _chan(m, fmt, entries):
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    ch = ComplexPolyphaseChannelizerM2(_taps(m, 9), 25000 * m, m, maxInputFloats=2 * MAX_BLOCKS * (m // 2))
    if fmt != "f32":
        ch.setSampleFormat(fmt)
    if entries is not None:
        ch.setOutputChannels(entries, _synth())
    return ch


def _update(ch, entries, prev, kept_two):
    """updateOutputChannels, with a new synthesis filter when no kept entry is a two-bin channel (else the current)"""
    ch.updateOutputChannels(entries, prev, None if kept_two else _synth())


# every bin corrected at gain M (pfb2_kernel's fused mix at M = 400 / 800), the paths test's mixed selection D (two-bin,
# corrected and plain one-bin channels, double gains), and every bin plain (the identity direct store)
KINDS = ["Cf", "D", "plain"]
CASES = [pytest.param(m, fmt, k, id="%d-%s-%s" % (m, fmt, k))
         for m, fmt in ((96, "f32"), (96, "u8"), (400, "f32"), (400, "u8"), (800, "f32"), (800, "u8")) for k in KINDS]


@pytest.mark.gpu
@pytest.mark.parametrize("m, fmt, kind", CASES)
def test_channel_rows_follow_the_oracle_through_selection_edits(gpu, m, fmt, kind):
    rng = np.random.default_rng(m + len(kind) + 3 * len(fmt))
    initial = [([b], 0, float(m)) for b in range(m)] if kind == "plain" else _selection(kind, m)
    raw, _ = _input(m, fmt)
    sizes = _calls(m, rng)
    need = 2 * sum(sizes)
    raw = np.concatenate([raw] * -(-need // raw.size))[:need]
    plan = _plan(initial, m, rng)

    res_chan, ch, still = _chan(m, fmt, None), _chan(m, fmt, initial), _chan(m, fmt, initial)
    cur = [Entry(idx, off, g, origin=j) for j, (idx, off, g) in enumerate(initial)]
    pos = 0
    for ci, n in enumerate(sizes):
        part = raw[pos:pos + 2 * n]
        pos += 2 * n
        if ci in plan:
            spec = plan[ci](cur)
            kept_two = any(p >= 0 and len(cur[p].idx) == 2 for p, _, _, _ in spec)
            cur, prev = _edit(cur, spec)
            _update(ch, [e.tuple() for e in cur], prev, kept_two)
        res = res_chan.receive(part)
        got = ch.receiveChannels(part)
        base = still.receiveChannels(part)
        assert got.shape == (len(cur), 2 * res.shape[0])
        bad = [i for i, e in enumerate(cur) if not np.array_equal(got[i], e.proc.process(res))]
        assert not bad, (ci, [(i, cur[i].idx) for i in bad[:4]])
        same = [(i, e.origin) for i, e in enumerate(cur) if e.origin is not None]
        assert np.array_equal(got[[i for i, _ in same]], base[[j for _, j in same]]), ci


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["Cf", "D"])
def test_an_update_with_every_entry_new_is_a_select(gpu, kind):
    """after some calls, an update in which every entry is -1 gives the rows sdrgpu_chan_select of the same channels
    gives, bit for bit, in every call that follows"""
    m, fmt = 400, "f32"
    rng = np.random.default_rng(5)
    initial = _selection(kind, m)
    raw, _ = _input(m, fmt)
    sizes = _calls(m, rng, 14)
    need = 2 * sum(sizes)
    raw = np.concatenate([raw] * -(-need // raw.size))[:need]
    target = [([b], int(rng.integers(-9000, 9000)), float(m)) for b in range(m)] if kind == "Cf" else \
        list(reversed(initial)) + [([7], 333, 1.5), ([m // 2 + 9, m // 2 + 10], -700, 2.0)]
    upd, sel = _chan(m, fmt, initial), _chan(m, fmt, initial)
    pos = 0
    for ci, n in enumerate(sizes):
        part = raw[pos:pos + 2 * n]
        pos += 2 * n
        if ci == 7:
            upd.updateOutputChannels(target, [-1] * len(target), _synth())
            sel.setOutputChannels(target, _synth())
        a, b = upd.receiveChannels(part), sel.receiveChannels(part)
        assert np.array_equal(a, b), ci


@pytest.mark.gpu
def test_refusals_change_nothing(gpu):
    """each refusal returns its code, and the rows that follow equal those of a channelizer that never received the
    refused call"""
    import ctypes as C
    from sdrtrunk_b200 import native
    L = gpu.lib()
    m = 96
    initial = _selection("D", m)
    x = np.random.default_rng(5).standard_normal(2 * 48 * 100).astype(np.float32) * 0.1
    ref, ch = _chan(m, "f32", initial), _chan(m, "f32", initial)
    half = 2 * 48 * 50
    want = [ref.receiveChannels(x[:half])]
    got = [ch.receiveChannels(x[:half])]
    keep = [(i, idx, off, g) for i, (idx, off, g) in enumerate(initial)]
    one = next(i for i, (idx, _, _) in enumerate(initial) if len(idx) == 1)
    two = next(i for i, (idx, _, _) in enumerate(initial) if len(idx) == 2)

    def call(spec, synth=None):
        arr = (native.OutputChannel * len(spec))(*[native.OutputChannel(int(idx[0]), int(idx[1]) if len(idx) == 2 else -1,
                                                                         int(off), float(g)) for _, idx, off, g in spec])
        prev = (C.c_int * len(spec))(*[p for p, _, _, _ in spec])
        f = None if synth is None else synth.ctypes.data_as(C.POINTER(C.c_float))
        return L.sdrgpu_chan_update_selection(ch._h, arr, prev, len(spec), f, 0 if synth is None else synth.size)

    def with_entry(i, entry):
        s = list(keep)
        s[i] = entry
        return s

    synth = np.ascontiguousarray(_synth(), np.float32)
    refused = [
        (with_entry(one, (one, [m], 0, float(m))), None),                       # bin out of range
        (with_entry(two, (two, [3, m + 1], 0, float(m))), None),                # second bin out of range
        (with_entry(one, (len(initial), [4], 0, float(m))), None),              # previous out of range
        (with_entry(one, (-2, [4], 0, float(m))), None),
        (keep + [(0,) + keep[0][1:]], None),                                    # an index named twice
        (with_entry(one, (one, [4, 5], 0, keep[one][3])), None),                # a kept entry changes class
        (with_entry(two, (two, [4], 0, keep[two][3])), None),
        (with_entry(one, (one, keep[one][1], 0, keep[one][3] * 2)), None),      # a kept entry changes gain
        (keep, synth),                                                          # a new filter with kept two-bin channels
    ]
    for spec, s in refused:
        assert call(spec, s) == gpu.ERR_INVALID_ARG, spec
    got.append(ch.receiveChannels(x[half:]))
    want.append(ref.receiveChannels(x[half:]))
    for g, w in zip(got, want):
        assert np.array_equal(g, w)

    # a new two-bin channel needs a filter when none was ever given; a corrected channel needs the sample rate
    plain = _chan(m, "f32", [([5], 0, float(m))])
    ch = plain
    assert call([(0, [5], 0, float(m)), (-1, [8, 9], 0, float(m))]) == gpu.ERR_INVALID_ARG
    h = C.c_void_p()
    t32 = np.ascontiguousarray(_taps(m, 9), np.float32)
    gpu.check(L.sdrgpu_chan_create(C.byref(h), t32.ctypes.data_as(C.POINTER(C.c_float)), t32.size, m, 1 << 16))

    class Raw:
        _h = h
    ch = Raw
    assert call([(5, [5], 300, float(m))]) == gpu.ERR_BAD_STATE
    assert call([(5, [5], 0, float(m)), (-1, [6], 0, float(m))]) == gpu.OK
    L.sdrgpu_chan_destroy(h)


@pytest.mark.gpu
def test_routed_pipeline_rows_follow_the_channelizer_through_edits(gpu):
    """a pipeline splitting the mixed selection over two pass-through banks (the ROUTED kernel instances) returns, after
    every edit that keeps the row count, the rows a channelizer alone returns; an edit that changes the row count gets
    BAD_STATE at the next pipeline call, and an edit back to the built count makes the pipeline usable again"""
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import Bank, Pipeline
    m, fmt = 400, "f32"
    rng = np.random.default_rng(11)
    initial = _selection("D", m)
    n_rows = len(initial)
    raw, _ = _input(m, fmt)
    sizes = [32 * (m // 2)] * 9    # within the input stream, whole blocks of the pass-through banks
    route = [int(r) for r in rng.integers(0, 2, n_rows)]
    route[:2] = [0, 1]
    banks = [Bank(route.count(j), CH_RATE, block_size=16, max_samples_per_call=2 * MAX_BLOCKS) for j in range(2)]
    routed_chan, alone = _chan(m, fmt, initial), _chan(m, fmt, initial)
    pipe = Pipeline(routed_chan, banks=banks, route=route)
    rev = lambda e: (list(reversed(e)), list(reversed(range(len(e)))))
    one = [i for i, e in enumerate(initial) if len(e[0]) == 1]
    two = [i for i, e in enumerate(initial) if len(e[0]) == 2]

    def retune(e):
        out = list(e)
        out[one[0]] = ([m // 2 + 40], 1234, e[one[0]][2])
        out[two[0]] = ([60, 61], e[two[0]][1], e[two[0]][2])
        return out, list(range(len(e)))

    def restart(e):
        return list(e), [-1 if i in (one[1], two[-1]) else i for i in range(len(e))]

    def grow(e):
        return list(e) + [([150], 77, 2.0)], list(range(len(e))) + [-1]

    def shrink(e):
        return list(e[:-1]), list(range(len(e) - 1))

    steps = {1: retune, 2: rev, 3: restart, 5: grow, 6: shrink, 7: rev}
    entries = list(initial)
    pos = 0
    for ci, n in enumerate(sizes):
        part = raw[2 * pos:2 * (pos + n)]
        if ci in steps:
            entries, prev = steps[ci](entries)
            for c in (routed_chan, alone):
                c.updateOutputChannels(entries, prev)
        if len(entries) != n_rows:
            with pytest.raises(native.IllegalStateException):
                pipe.process(part)
            continue
        pos += n
        out = pipe.process(part)
        want = alone.receiveChannels(part)
        rows = np.empty_like(want)
        for j in range(2):
            rows[[i for i in range(n_rows) if route[i] == j]] = out[j]
        assert np.array_equal(rows, want), ci
    pipe.dispose()


@pytest.mark.gpu
def test_selection_edits_through_the_pipeline_schedules(gpu):
    """Two tuners feed a C4FM bank; edits that keep the row count (retune a channel to another bin, reverse the order,
    restart one in place, change offsets with the edit) land between calls.  The dibits are identical through the
    single pass, the filters-first schedule on device input, submit / wait with the edit issued while two calls are in
    flight (applied from the next submit), and the reference sequence receiveChannels -> Bank.process."""
    import ctypes as C
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
    # per call: {tuner: (entries, previous)}
    plan = {1: {0: ([([2], 37), ([40], -53), ([77], 120)], [0, 1, 2]), 1: ([([95], 0), ([6], 9), ([5], -200)], [2, 1, 0])},
            2: {0: ([([2], 37), ([30], -310), ([77], 120)], [0, 1, -1])},
            3: {1: ([([95], 0), ([6], 250), ([5], -200)], [0, -1, 2])},
            4: {0: ([([77], 0), ([30], -310), ([2], 400)], [2, 1, 0]), 1: ([([5], -200), ([6], 250), ([95], 75)], [2, 1, 0])},
            5: {0: ([([77], 61), ([30], -310), ([2], 400)], [0, 1, 2])}}

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
        for k, (entries, prev) in plan.get(i, {}).items():
            cs[k].updateOutputChannels(entries, prev)

    single, cs = pipeline(1)
    want = []
    for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
        apply(cs, i)
        want.append(single.process([x[a:b] for x in xs]))
    assert sum(w.size for w in want[2]) > 1000

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
