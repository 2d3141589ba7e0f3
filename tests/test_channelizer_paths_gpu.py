"""Every output path of the CUDA channelizer against a float64 reference and against each other.

Which kernel instance runs depends on the channel count M (a pfb2_kernel row of kPfbRows, or pfb_ifft_kernel with 8- or
16-block tiles and 9 or any other number of taps per channel), the input format (8-bit samples read as they are by the
M = 400 / 800 rows), the selection (every bin, a subset, frequency-corrected or two-bin channels, float or double gains)
and whether a pipeline stores the rows through its row table (the ROUTED instances).  Each case below runs one stream
through one of them, in ragged calls that reach the framing edges, and checks

1. bit for bit: every channel row equals the same channelizer's results-layout column through the output stage
   (gain product, Oscillator mix + applyGain, TwoChannelOutputProcessor); 8-bit input equals the converted floats;
2. every row of every output against a float64 reference: the oracle's float32 filter-bank accumulators (bit-exact with
   the CUDA filter bank) through a float64 inverse DFT.  The only legitimate difference is the rounding of the float32
   inverse DFT, so each row's RMS error must stay below TOL times the RMS of all rows of the stream;
3. bit for bit: a pipeline that splits the rows over two pass-through banks gives every row the unrouted call gave.
"""
import ctypes as C
import functools

import numpy as np
import pytest

import oracle
import siggen as sg

CH_RATE = 50000.0   # 25 kHz bins, 2x oversampled
TOL = 1e-6          # per-row RMS error against the float64 reference, relative to the RMS of all rows

# ragged calls, in units of M/2 complex samples (+ extra samples): a first call shorter than the history (its tiles read
# the zero history: the !fast filter-bank path), fewer blocks than one tile, a call that completes no block, an odd
# block count that is no multiple of the tile (parity flip), a long call (many CTAs; the one that saves the history is
# not CTA 0) and the rest
CALLS = ((3, 7), (5, 0), (0, 10), (37, 3), (300, 0), (11, 5))
N_BLOCKS = 356      # blocks the calls above complete


def white(rng, n):
    return sg.interleave(sg.awgn(rng, n, 0.1))


def reference(taps, m, x):
    """float64 channelizer results, complex [n_blocks, M] (numpy's ifft includes the 1/M)"""
    raw = oracle.Channelizer(taps, m).receive(x, mode="raw").astype(np.float64)
    return np.fft.ifft(raw[:, 0::2] + 1j * raw[:, 1::2], axis=1)


def interleaved(z):
    """complex [n_blocks, M] -> float32 results layout [n_blocks, 2M]"""
    out = np.empty((z.shape[0], 2 * z.shape[1]), np.float32)
    out[:, 0::2] = z.real
    out[:, 1::2] = z.imag
    return out


def bin_rows(res, m):
    """results layout [n_blocks, 2M] -> one interleaved row per bin [M, 2 n_blocks]"""
    return res.reshape(res.shape[0], m, 2).transpose(1, 0, 2).reshape(m, -1)


def row_errors(got, want, scale):
    """RMS error of each row of got / want ([rows, n] float arrays) over `scale`"""
    d = np.asarray(got, np.float64) - np.asarray(want, np.float64)
    return np.sqrt(np.mean(d ** 2, axis=1)) / scale


# ------------------------------------------------------------------------------------------ the reference, without a GPU
@pytest.mark.parametrize("m", [2, 70, 96, 114, 400, 800])
def test_float64_reference_matches_oracle_f64_mode(m):
    """the numpy inverse DFT over the oracle's float32 accumulators is the oracle's float64 channelizer, every row"""
    rng = np.random.default_rng(m)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9) if m > 2 else np.hanning(18).astype(np.float32)
    x = white(rng, m // 2 * 60 + m // 4)
    got = interleaved(reference(taps, m, x))
    want = oracle.Channelizer(taps, m).receive(x, mode="f64")
    assert got.shape == want.shape == (60, 2 * m)
    scale = np.sqrt(np.mean(want.astype(np.float64) ** 2))
    assert row_errors(bin_rows(got, m), bin_rows(want, m), scale).max() <= 1e-7


@pytest.mark.parametrize("m", [96, 400])
def test_float64_reference_tone_lands_in_its_bin(m):
    """a tone at bin k + df comes out of row k at its amplitude, rotating by df per channel sample"""
    k, df, amp = 7, 2000.0, 0.25
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    x = sg.interleave(sg.tone(25000.0 * m, k * 25000.0 + df, m // 2 * 400, amplitude=amp))
    z = reference(taps, m, x)[40:] * m                       # gain M, as OneChannelOutputProcessor
    power = np.mean(np.abs(z) ** 2, axis=0)
    assert power.argmax() == k
    assert abs(np.sqrt(power[k]) - amp) < 1e-3
    step = np.angle(np.mean(z[1:, k] * np.conj(z[:-1, k])))
    assert abs(step - 2 * np.pi * df / CH_RATE) < 1e-5


# ------------------------------------------------------------------------------------------------------ GPU cases
# (M, taps per channel, input format): every pfb2_kernel row of kPfbRows on float input, its 8-bit instances (M = 400 /
# 800), 16-bit input converted in front of a row with 8-bit instances, and the four pfb_ifft_kernel instances: 16-block
# tiles (M = 114 = 2 x 3 x 19, M = 96 with a T = 5 prototype) and 8-block tiles (M = 480), each with T = 9 and a run-time T
ROWS = [(m, 9, "f32") for m in (400, 800, 96, 640, 320, 240, 200, 160, 120, 100, 80)]
RAW = [(400, 9, "u8"), (400, 9, "s8"), (800, 9, "u8"), (800, 9, "s8")]
GENERIC = [(114, 9, "f32"), (96, 5, "f32"), (480, 9, "f32"), (480, 5, "f32")]

# A: the default selection (every bin, gain M); B: a shuffled subset with float gains, Bd: the same with one gain that is
# no float (every row on the double path); Cf / Cd: every bin frequency-corrected at gain M / at a double gain; D: two-bin
# channels on adjacent bins (across the middle and at the top), corrected and plain one-bin channels, double gains
SELECTIONS = ["A", "B", "Bd", "Cf", "Cd", "D"]
CASES = ([pytest.param(c, s, id="%d-T%d-%s-%s" % (c + (s,))) for c in ROWS + GENERIC for s in SELECTIONS] +
         [pytest.param(c, s, id="%d-T%d-%s-%s" % (c + (s,))) for c in RAW for s in ("A", "Cf", "Cd", "D")] +
         [pytest.param((800, 9, "s16le"), s, id="800-T9-s16le-%s" % s) for s in ("A", "D")])


def _taps(m, t):
    return oracle.sinc_m2_channelizer(25000.0, m, t)


def _synth():
    return oracle.sinc_m2_synthesizer(CH_RATE, 25000.0, 2, 9)


def _input(m, fmt):
    """one stream of white samples in the tuner format: (raw values, the float32 samples they convert to)"""
    rng = np.random.default_rng(m + 7 * len(fmt))
    n = sum(b * (m // 2) + e for b, e in CALLS)
    if fmt == "f32":
        x = white(rng, n)
        return x, x
    raw = {"u8": lambda: rng.integers(0, 256, 2 * n, dtype=np.uint8),
           "s8": lambda: rng.integers(-128, 128, 2 * n, dtype=np.int8),
           "s16le": lambda: rng.integers(-32768, 32768, 2 * n).astype("<i2")}[fmt]()
    return raw, oracle.convert_samples(raw.tobytes(), fmt)


def _calls(m, x):
    pos = 0
    for b, e in CALLS:
        n = 2 * (b * (m // 2) + e)
        yield x[pos:pos + n]
        pos += n
    assert pos == x.size


def _channelizer(m, t, fmt, entries=None):
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    ch = ComplexPolyphaseChannelizerM2(_taps(m, t), 25000 * m, m)
    if fmt != "f32":
        ch.setSampleFormat(fmt)
    if entries is not None:
        ch.setOutputChannels(entries, _synth())
    return ch


@functools.lru_cache(maxsize=None)
def _results(m, t, fmt):
    """(GPU results layout over the ragged calls, float64 reference, worst per-row error of the results layout)"""
    raw, x = _input(m, fmt)
    ch = _channelizer(m, t, fmt)
    res = np.concatenate([ch.receive(part) for part in _calls(m, raw)])
    assert res.shape == (N_BLOCKS, 2 * m)
    if fmt != "f32":
        # 8-bit samples read by the filter bank (16-bit: converted first) == the converted floats, bit for bit
        f = _channelizer(m, t, "f32")
        assert np.array_equal(res, np.concatenate([f.receive(part) for part in _calls(m, x)]))
    ref = reference(_taps(m, t), m, x)
    scale = float(np.sqrt(np.mean(np.abs(ref) ** 2) / 2))    # RMS of the I and Q values of all rows
    err = row_errors(bin_rows(res, m), bin_rows(interleaved(ref), m), scale)
    print("\nchannelizer M = %d, T = %d, %s: worst per-row error against float64 %.3g (row %d)" %
          (m, t, fmt, err.max(), err.argmax()))
    return res, ref, float(err.max())


def _gain_product(v, g):
    """applyGain: (float)(v * (double)g); for a float gain the same as one float product"""
    if float(np.float32(g)) == g:
        return (np.asarray(v, np.float32) * np.float32(g)).astype(np.float32)
    return (np.asarray(v, np.float64) * g).astype(np.float32)


def _output_stage(res, entries):
    """the rows of `entries` computed from results-layout rows `res` by the oracle's output processors"""
    out = []
    for idx, off, g in entries:
        if len(idx) == 2:
            p = oracle.TwoChannelOutputProcessor(CH_RATE, idx[0], idx[1], _synth(), g)
            p.set_frequency_offset(off)
            out.append(p.process(res))
            continue
        v = np.ascontiguousarray(res[:, 2 * idx[0]:2 * idx[0] + 2]).ravel()
        out.append(oracle.apply_gain(oracle.Oscillator(off, CH_RATE).mix(v), g) if off else _gain_product(v, g))
    return np.array(out)


def _selection(kind, m):
    """setOutputChannels entries (indexes, frequency offset, gain); None for the default selection"""
    rng = np.random.default_rng(m + ord(kind[0]))
    if kind == "A":
        return None
    if kind in ("B", "Bd"):
        edges = [0, m // 2 - 1, m // 2, m - 1]
        bins = edges + [int(b) for b in rng.choice([b for b in range(m) if b not in edges], 12, replace=False)]
        bins = [bins[i] for i in rng.permutation(len(bins))]
        gains = [(1.0, 2.5, float(m), 0.75, 1.0 / 64)[i % 5] for i in range(len(bins))]
        if kind == "Bd":
            gains[5] = 0.1
        return [([b], 0, g) for b, g in zip(bins, gains)]
    if kind in ("Cf", "Cd"):
        offsets = [int(v) for v in rng.integers(-12000, 12000, m)]
        offsets[3] = 1
        return [([b], offsets[b], float(m) if kind == "Cf" else 0.1) for b in range(m)]
    return [([m // 2 - 1, m // 2], -2500, float(m)), ([3], 900, float(m)), ([m - 2, m - 1], 0, float(m)), ([20], 0, 2.5),
            ([10, 11], 1500, 1.0 / 3), ([m // 2 + 3], -4321, 1.0 / 3), ([0], 0, float(m)), ([m // 2 + 5], 0, 0.1),
            ([m - 5], 6250, float(m))]


def _entries(kind, m):
    sel = _selection(kind, m)
    return [([b], 0, float(m)) for b in range(m)] if sel is None else sel


def _routed(m, t, fmt, sel, raw, n_rows, device_input):
    """the rows of a pipeline that splits the selection over two pass-through banks (no FIR, no demodulator), gathered
    back into selection order; host input in the ragged calls, or device input in one call"""
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import Bank, Pipeline
    route = [int(r) for r in np.random.default_rng(n_rows).integers(0, 2, n_rows)]
    route[:2] = [0, 1]
    banks = [Bank(route.count(j), CH_RATE, block_size=16, max_samples_per_call=2 * N_BLOCKS) for j in range(2)]
    pipe = Pipeline(_channelizer(m, t, fmt, sel), banks=banks, route=route)
    if device_input:
        L = native.lib()
        d = C.c_void_p()
        native.check(L.sdrgpu_device_alloc(C.byref(d), raw.nbytes))
        native.check(L.sdrgpu_memcpy(d, native.ptr(raw), raw.nbytes, native.DEVICE, native.HOST))
        parts = [pipe.process(d.value, native.DEVICE, raw.size)]
        L.sdrgpu_device_free(d)
    else:
        parts = [pipe.process(part) for part in _calls(m, raw)]
    pipe.dispose()
    per_bank = [np.concatenate([p[j] for p in parts], axis=1) for j in range(2)]
    n = per_bank[0].shape[1]
    assert n == per_bank[1].shape[1] == 2 * (N_BLOCKS // 16 * 16)
    rows = np.empty((n_rows, n), np.float32)
    for j in range(2):
        rows[[i for i in range(n_rows) if route[i] == j]] = per_bank[j]
    return rows


@pytest.mark.gpu
def test_pass_through_bank_returns_its_input(gpu):
    """the banks the routed checks use: no decimation, no FIR, no demodulator -- their rows come back unchanged"""
    from sdrtrunk_b200.dsp import Bank
    x = np.random.default_rng(3).standard_normal((3, 2 * 80)).astype(np.float32)
    bank = Bank(3, CH_RATE, block_size=16, max_samples_per_call=256)
    assert np.array_equal(bank.process(x), x)


@pytest.mark.gpu
@pytest.mark.parametrize("case, kind", CASES)
def test_channel_rows_bit_exact_and_within_float64_bound(gpu, case, kind):
    m, t, fmt = case
    res, ref, worst = _results(m, t, fmt)
    assert worst <= TOL, (m, t, fmt, worst)
    raw, _ = _input(m, fmt)
    sel = _selection(kind, m)
    entries = _entries(kind, m)
    ch = _channelizer(m, t, fmt, sel)
    got = np.concatenate([ch.receiveChannels(part) for part in _calls(m, raw)], axis=1)
    assert got.shape == (len(entries), 2 * N_BLOCKS)

    # 1. the channel rows are the results layout through the output stage, bit for bit
    want = _output_stage(res, entries)
    bad = [i for i in range(len(entries)) if not np.array_equal(got[i], want[i])]
    assert not bad, [entries[i] for i in bad[:4]]

    # 2. every row within TOL of the float64 reference through the same output stage
    want64 = _output_stage(interleaved(ref), entries)
    scale = float(np.sqrt(np.mean(np.abs(ref) ** 2) / 2))
    err = row_errors(got, want64, scale * np.array([abs(g) for _, _, g in entries]))
    assert err.max() <= TOL, (entries[int(err.argmax())], float(err.max()))

    # 3. a pipeline's row table (the ROUTED instances) stores the same rows, from host and from device input
    for device_input in (False, True):
        rows = _routed(m, t, fmt, sel, raw, len(entries), device_input)
        assert np.array_equal(rows, got[:, :rows.shape[1]]), device_input
