"""Parity of the CUDA polyphase channelizer (through the C ABI) against the oracle.

Tolerance here: 1e-4 relative RMS per channel (BASELINE.json north_star; the inverse DFT's summation order differs
from JTransforms' by construction).  The filter-bank stage itself is arithmetic-identical (products rounded,
sequential adds), so the only legitimate difference is the rounding of the float32 inverse DFT, ~1e-7:
test_channelizer_paths_gpu.py holds every row of every kernel instance to 1e-6 of the RMS of all rows against a
float64 reference (the oracle's float32 filter-bank accumulators through a float64 inverse DFT).
"""
import numpy as np
import pytest

import oracle
import siggen as sg

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _signal(rng, n, m):
    """random-phase tones near a handful of bin centres + AWGN, amplitude in the tuner's [-1, 1] range"""
    fs = 25000.0 * m
    z = sg.awgn(rng, n, 1e-3)
    for k in rng.choice(m, size=min(m, 12), replace=False):
        f = (k if k < m // 2 else k - m) * 25000.0 + rng.uniform(-5000, 5000)
        z = z + sg.tone(fs, f, n, amplitude=0.05, phase=rng.uniform(0, 2 * np.pi))
    return sg.interleave(z)


@pytest.mark.parametrize("m", [96, 400, 800, 114, 70, 2, 80, 100, 120, 160, 200, 240, 320, 640])
def test_results_layout_matches_oracle(gpu, m):
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    rng = np.random.default_rng(m)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9) if m > 2 else np.hanning(18).astype(np.float32)
    x = _signal(rng, 37 * m // 2 + 5, m)
    want = oracle.Channelizer(taps, m).receive(x, mode="f64")
    ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
    got = ch.receive(x)
    assert got.shape == want.shape
    assert sg.rel_rms(got, want) < TOL
    # per-bin check on the bins that carry signal
    power = np.sum(want.reshape(want.shape[0], m, 2) ** 2, axis=(0, 2))
    for k in np.argsort(power)[-4:]:
        assert sg.rel_rms(got[:, 2 * k:2 * k + 2], want[:, 2 * k:2 * k + 2]) < TOL


@pytest.mark.parametrize("m", [96, 400, 800, 100, 320, 640, 80, 120, 160, 200, 240])
def test_channel_layout_matches_oracle_output_processor(gpu, m):
    """m = 800 is BASELINE configs[4]'s channel count (pfb2_kernel<800, 32, 25>: odd second factor, direct row stores)"""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    rng = np.random.default_rng(100 + m)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    x = _signal(rng, 53 * m // 2, m)
    res = oracle.Channelizer(taps, m).receive(x, mode="f64")
    ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
    got = ch.receiveChannels(x)                       # default selection: all bins, gain M
    assert got.shape == (m, 2 * res.shape[0])
    # every bin against the oracle's output processor: a store that lands in the wrong row cannot hide
    rows = range(m) if m == 800 else (0, 1, m // 2 - 1, m // 2, m - 1)
    wants = {k: oracle.OneChannelOutputProcessor(50000.0, k, float(m)).process(res) for k in rows}
    rms = {k: float(np.sqrt(np.mean(wants[k].astype(np.float64) ** 2))) for k in rows}
    scale = max(rms.values())
    for k in rows:
        err = float(np.sqrt(np.mean((got[k].astype(np.float64) - wants[k]) ** 2)))
        assert err < TOL * scale, k                    # absolute, against the strongest bin (noise-only bins too)
        if rms[k] > 0.1 * scale:                       # bins that carry a tone: relative per bin
            assert sg.rel_rms(got[k], wants[k]) < TOL, k
    # explicit selection of a subset, in caller order
    bins = [5, m - 2, 0, 17]
    ch2 = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
    ch2.setChannels(bins)
    sub = ch2.receiveChannels(x)
    assert sub.shape == (4, 2 * res.shape[0])
    assert np.array_equal(sub, got[bins])


def test_streaming_framing_is_independent_of_buffer_length(gpu):
    """mSampleBufferPointer carry-over (ComplexPolyphaseChannelizerM2.java:202-227): ragged / tiny / empty buffers"""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m = 96
    rng = np.random.default_rng(7)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    x = _signal(rng, 6000, m)
    whole = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m).receive(x)
    ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
    parts, pos = [], 0
    for n in (2, 0, 94, 96, 1000, 98, 3710, 7000):
        parts.append(ch.receive(x[pos:pos + n]))
        pos += n
    assert pos == x.size
    got = np.concatenate(parts)
    assert got.shape == whole.shape
    assert np.array_equal(got, whole)                 # same arithmetic regardless of framing
    want = oracle.Channelizer(taps, m).receive(x, mode="f64")
    assert sg.rel_rms(got, want) < TOL


def test_filter_bank_stage_is_bit_exact_on_dc_bin(gpu):
    """Bin 0 of the inverse DFT is the plain sum of the filter-bank accumulators; feeding a signal that only
    excites one polyphase branch makes that sum a single term, which must match the oracle's accumulators."""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m = 96
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    x = np.zeros(2 * 48 * 40, np.float32)
    x[2 * 17::2 * 48] = np.random.default_rng(8).standard_normal(40).astype(np.float32)   # one branch only
    raw = oracle.Channelizer(taps, m).receive(x, mode="raw")
    got = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m).receive(x)
    want0 = raw.reshape(raw.shape[0], m, 2).sum(axis=1) * np.float32(1.0 / m)
    assert np.array_equal(got[:, 0:2], want0.astype(np.float32))


def test_custom_taps_per_channel_generic_path(gpu):
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m = 40
    rng = np.random.default_rng(9)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 5)   # T = 5 -> runtime-T filter-bank path
    x = _signal(rng, 3000, m)
    want = oracle.Channelizer(taps, m).receive(x, mode="f64")
    got = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m).receive(x)
    assert sg.rel_rms(got, want) < TOL


@pytest.mark.parametrize("seed", range(8))
def test_random_channel_counts_and_taps_per_channel(gpu, seed):
    """generic kernel: channel counts with every kind of factorisation (powers of two, 3s, 5s, large primes), taps per
    channel other than the reference's 9, random prototypes, ragged buffers"""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    rng = np.random.default_rng(1000 + seed)
    m = int(rng.choice([4, 6, 14, 22, 34, 46, 62, 74, 128, 134, 250, 256, 358, 486, 514, 1000]))
    t = int(rng.choice([1, 2, 3, 5, 9, 12]))
    taps = (rng.standard_normal(m * t) / (m * t)).astype(np.float32)
    n = (10 + int(rng.integers(0, 40))) * (m // 2) + int(rng.integers(0, m // 2))
    x = sg.interleave(rng.standard_normal(n) + 1j * rng.standard_normal(n))
    want = oracle.Channelizer(taps, m).receive(x, mode="f64")
    ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
    cut = 2 * int(rng.integers(0, n))
    got = np.concatenate([ch.receive(x[:cut]), ch.receive(x[cut:])])
    assert got.shape == want.shape, (m, t)
    assert sg.rel_rms(got, want) < TOL, (m, t)


def test_errors_mirror_reference(gpu):
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    with pytest.raises(native.IllegalArgumentException):
        ComplexPolyphaseChannelizerM2(np.ones(27, np.float32), 75000, 3)     # odd channel count (:97-100)
    ch = ComplexPolyphaseChannelizerM2(1e6, 9, maxInputFloats=4096)          # designs its own prototype (:114-126)
    assert ch.mChannelCount == 40 and ch.mTapsPerChannel == 9
    with pytest.raises(native.IllegalArgumentException):
        ch.receive(np.zeros(7, np.float32))                                   # odd float count
    with pytest.raises(native.OverflowError_):
        ch.receive(np.zeros(8192, np.float32))
    with pytest.raises(native.IllegalArgumentException):
        ch.setChannels([40])


def test_full_size_tone_property(gpu):
    """BASELINE config 2 size: 10 MS/s -> 400 channels, one TestTuner buffer of 500 000 samples; a tone placed
    at bin k + df lands in channel k at unit amplitude rotating at df (size-independent property)."""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m, fs, n = 400, 1e7, 500000
    ch = ComplexPolyphaseChannelizerM2(fs, 9)
    k, df = 123, 2500.0
    z = sg.tone(fs, k * 25000.0 + df, n, amplitude=0.25)
    out = ch.receiveChannels(sg.interleave(z))
    assert out.shape == (m, 2 * (n // 200))
    power = np.mean(out[:, 200:] ** 2, axis=1) * 2
    assert power.argmax() == k
    assert abs(np.sqrt(power[k]) - 0.25) < 1e-3
    others = np.delete(power, [k - 1, k, k + 1])
    assert others.max() < 1e-7 * power[k] * 1e2          # >= 50 dB down outside the adjacent bins
    c = sg.deinterleave(out[k, 200:])
    step = np.angle(np.mean(c[1:] * np.conj(c[:-1])))
    assert abs(step - 2 * np.pi * df / 50000.0) < 1e-4


def test_device_resident_io(gpu):
    """SDRGPU_DEVICE pointers in and out: no host copies inside the call."""
    import ctypes as C
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m = 96
    rng = np.random.default_rng(10)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    x = _signal(rng, 4800, m)
    host = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m).receiveChannels(x)
    ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
    L = native.lib()
    d_in, d_out = C.c_void_p(), C.c_void_p()
    native.check(L.sdrgpu_device_alloc(C.byref(d_in), x.nbytes))
    native.check(L.sdrgpu_device_alloc(C.byref(d_out), host.nbytes))
    native.check(L.sdrgpu_memcpy(d_in, native.ptr(x), x.nbytes, native.DEVICE, native.HOST))
    nb = ch.receiveChannels((d_in.value, x.size), native.DEVICE, d_out.value, native.DEVICE, host.shape[1])
    ch.sync()
    back = np.empty_like(host)
    native.check(L.sdrgpu_memcpy(native.ptr(back), d_out, host.nbytes, native.HOST, native.DEVICE))
    assert nb == host.shape[1] // 2
    assert np.array_equal(back, host)
    L.sdrgpu_device_free(d_in)
    L.sdrgpu_device_free(d_out)


def test_frequency_offset_and_two_channel_output_processors(gpu):
    """a6 / a7: OneChannelOutputProcessor with the frequency-correction Oscillator and TwoChannelOutputProcessor
    (TwoChannelSynthesizerM2 + FS4DownConverter + Oscillator) against the oracle, fed the oracle's own float32
    channelizer results re-created by the GPU channelizer (the rows differ only by the inverse DFT's rounding, so the
    comparison is at the 1e-4 relative-RMS bar), across ragged calls (state carried: oscillator, serpentine, fs/4)."""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m, fs = 96, 2.4e6
    rng = np.random.default_rng(21)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    synth = oracle.sinc_m2_synthesizer(50000.0, 25000.0, 2, 9)
    n = 48 * 700
    z = sg.awgn(rng, n, 1e-3)
    z = z + sg.tone(fs, 7 * 25000.0 + 900.0, n, 0.2) + sg.tone(fs, 20 * 25000.0 + 12500.0 - 2500.0, n, 0.3)
    z = z + sg.tone(fs, -5 * 25000.0 - 12500.0 + 4000.0, n, 0.25)      # straddles bins 90 / 91
    x = sg.interleave(z)
    res = oracle.Channelizer(taps, m).receive(x, mode="f64")

    ch = ComplexPolyphaseChannelizerM2(taps, int(fs), m)
    ch.setOutputChannels([([7], 900), ([20, 21], -2500), ([3], 0), ([90, 91], 0), ([40], -1234, 2.5)], synth)
    parts, pos = [], 0
    for cut in (2 * 48 * 100, 2 * 48 * 33 + 10, 2 * 48 * 300, x.size):
        cut = min(cut + pos, x.size)
        parts.append(ch.receiveChannels(x[pos:cut]))
        pos = cut
    got = np.concatenate(parts, axis=1)
    assert got.shape == (5, 2 * res.shape[0])

    one = oracle.OneChannelOutputProcessor(50000.0, 7, float(m))
    one.set_frequency_offset(900)
    two = oracle.TwoChannelOutputProcessor(50000.0, 20, 21, synth, float(m))
    two.set_frequency_offset(-2500)
    plain = oracle.OneChannelOutputProcessor(50000.0, 3, float(m))
    two0 = oracle.TwoChannelOutputProcessor(50000.0, 90, 91, synth, float(m))
    one_g = oracle.OneChannelOutputProcessor(50000.0, 40, 2.5)
    one_g.set_frequency_offset(-1234)
    want = [one.process(res), two.process(res), plain.process(res), two0.process(res), one_g.process(res)]
    for i in range(5):
        assert sg.rel_rms(got[i], want[i]) < TOL, i
    # the corrected one-bin channel: the 900 Hz residual is mixed to DC (Oscillator conjugate rotation at -900 Hz ...)
    c = sg.deinterleave(want[0][200:])
    assert abs(np.angle(np.mean(c[1:] * np.conj(c[:-1])))) < 2 * np.pi * 2000 / 50000.0
    # errors as the Java: more than two indexes / synthesis filter missing
    from sdrtrunk_b200 import native
    with pytest.raises(native.IllegalArgumentException):
        ch.setOutputChannels([([1, 2, 3], 0)])


def test_frequency_corrected_channels_oscillator_look_ahead_is_bit_exact(gpu):
    """One-bin channels with an offset take their oscillator values from a ring that a side-stream kernel fills ahead of
    use.  Fed the GPU's own uncorrected rows, the oracle's Oscillator + applyGain must reproduce every corrected row bit
    for bit, across many ragged calls (ring wrap-around, calls longer than the look-ahead left in the ring, empty calls)."""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m, fs = 96, 2.4e6
    rng = np.random.default_rng(23)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    n = 48 * 3000
    x = sg.interleave(sg.awgn(rng, n, 0.1))
    bins_offsets = [(7, 900), (3, -12000), (50, 1), (95, 6250), (20, -3333)]
    max_floats = 2 * 48 * 400                              # look-ahead of 400 blocks: the stream below wraps it many times
    plain = ComplexPolyphaseChannelizerM2(taps, int(fs), m, maxInputFloats=max_floats)
    plain.setChannels([b for b, _ in bins_offsets], gain=1.0)
    corr = ComplexPolyphaseChannelizerM2(taps, int(fs), m, maxInputFloats=max_floats)
    corr.setOutputChannels([([b], off, 96.0) for b, off in bins_offsets])
    oscs = [oracle.Oscillator(off, 50000.0) for _, off in bins_offsets]
    pos = 0
    sizes = [400, 1, 399, 400, 0, 17, 400, 250, 400, 400, 83]
    while pos < n:
        for blocks in sizes:
            cut = min(x.size, 2 * (pos + 48 * blocks))
            rows = plain.receiveChannels(x[2 * pos:cut])
            got = corr.receiveChannels(x[2 * pos:cut])
            for i, o in enumerate(oscs):
                want = oracle.apply_gain(o.mix(rows[i]), 96.0)
                assert np.array_equal(got[i], want), (pos, i)
            pos = cut // 2
            if pos >= n:
                break


@pytest.mark.parametrize("m", [96, 160, 400, 800])
def test_every_bin_frequency_corrected_is_mixed_in_the_channelizer_kernel(gpu, m):
    """all M bins selected in order as frequency-corrected one-bin channels with one gain: a pfb2_kernel instance with
    8-block tiles (M = 160 ... 800) multiplies the look-ahead oscillator values in where it stores the rows (no
    osc_mix_kernel pass); one with 16-block tiles (M = 96) leaves them to osc_mix_kernel.  Every row must equal the
    oracle's Oscillator + applyGain on the GPU's own uncorrected row, bit for bit, across ragged calls that wrap the rings."""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    fs = 25000.0 * m
    rng = np.random.default_rng(29)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    half = m // 2
    n = half * 900
    x = sg.interleave(sg.awgn(rng, n, 0.1))
    offsets = [int(v) for v in rng.integers(-12000, 12000, m)]
    offsets[3] = 1
    max_floats = 2 * half * 200
    plain = ComplexPolyphaseChannelizerM2(taps, int(fs), m, maxInputFloats=max_floats)
    plain.setChannels(list(range(m)), gain=1.0)
    corr = ComplexPolyphaseChannelizerM2(taps, int(fs), m, maxInputFloats=max_floats)
    corr.setOutputChannels([([b], offsets[b], float(m)) for b in range(m)])
    check = sorted({0, 1, 3, 19, 20, m // 2 - 1, m // 2, m - 2, m - 1} | set(int(v) for v in rng.integers(0, m, 24)))
    oscs = {b: oracle.Oscillator(offsets[b], 50000.0) for b in check}
    pos = 0
    for blocks in [200, 1, 199, 8, 0, 7, 200, 85, 200]:
        cut = min(x.size, 2 * (pos + half * blocks))
        rows = plain.receiveChannels(x[2 * pos:cut])
        got = corr.receiveChannels(x[2 * pos:cut])
        for b in check:
            want = oracle.apply_gain(oscs[b].mix(rows[b]), float(m))
            assert np.array_equal(got[b], want), (pos, b)
        pos = cut // 2
    assert pos == n


@pytest.mark.parametrize("m", [96, 400, 800])
@pytest.mark.parametrize("fmt", ["u8", "s8", "s16le"])
def test_native_tuner_sample_formats(gpu, fmt, m):
    """section 8f #1: ByteSampleConverter / SignedByteSampleConverter / 16-bit conversion on the device, standalone
    (bit-exact: integer / power of two, or one correctly rounded division) and fused in front of the channelizer.  For
    M = 400 / 800 the filter bank itself reads the 8-bit samples (no float copy of the input): ragged calls cover its
    tiles that reach into the float history, a call shorter than one block (converted by the stand-alone kernel) and the
    history the kernel saves from raw samples."""
    from sdrtrunk_b200.dsp import (ByteSampleConverter, ComplexPolyphaseChannelizerM2, Signed16BitSampleConverter,
                                   SignedByteSampleConverter)
    rng = np.random.default_rng(31)
    n = m // 2 * 300
    if fmt == "u8":
        raw = rng.integers(0, 256, 2 * n, dtype=np.uint8)
        conv = ByteSampleConverter()
    elif fmt == "s8":
        raw = rng.integers(-128, 128, 2 * n, dtype=np.int8)
        conv = SignedByteSampleConverter()
    else:
        raw = rng.integers(-32768, 32768, 2 * n).astype("<i2")
        conv = Signed16BitSampleConverter()
    want_f = oracle.convert_samples(raw.tobytes(), fmt)
    assert np.array_equal(conv.convertSamples(raw.tobytes()), want_f)
    edge = {"u8": np.array([0, 127, 128, 255], np.uint8), "s8": np.array([-128, -1, 0, 127], np.int8),
            "s16le": np.array([-32768, -1, 0, 32767], "<i2")}[fmt]
    assert np.array_equal(conv.convertSamples(edge.tobytes()), oracle.convert_samples(edge.tobytes(), fmt))
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
    ch.setSampleFormat(fmt)
    got = np.concatenate([ch.receive(raw[:10000]), ch.receive(raw[10000:10050]), ch.receive(raw[10050:10050 + 34 * m]),
                          ch.receive(raw[10050 + 34 * m:])])
    ref = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m).receive(want_f)       # same kernels on converted floats
    assert np.array_equal(got, ref)
    assert sg.rel_rms(got, oracle.Channelizer(taps, m).receive(want_f, mode="f64")) < TOL


# ------------------------------------------------------------------------------------------------ Airspy raw samples
@pytest.mark.parametrize("packed", [False, True])
def test_airspy_sample_converter_bit_exact(gpu, packed):
    """AirspySampleConverter on the device: unpack + DCRemovalFilter + HilbertTransform, every float equal to the
    oracle's.  The DC recursion is sequential; the device runs it speculatively per 4 096-sample segment and verifies,
    so long buffers (many segments), short ones, odd cuts and a stream with a large DC step are all covered."""
    from sdrtrunk_b200.dsp import AirspySampleConverter
    rng = np.random.default_rng(5 + packed)
    n = 300000
    x = sg.airspy_real_signal(rng, n, [(1.3e6, 0.3), (-2.2e6, 0.1)], dc=0.03)
    x[150000:] += 0.2                                     # DC jump in the middle of the stream
    raw = sg.airspy_raw(x, packed)
    bps = 3 if packed else 4                              # bytes per pair of samples
    ref = oracle.AirspySampleConverter()
    ref.setSamplePacking(packed)
    conv = AirspySampleConverter(maxSamples=1 << 18)
    conv.setSamplePacking(packed)
    pos = 0
    for pairs in (100000, 1, 23, 3000, 2048, 2049, 0, 40000):       # in pairs of samples
        chunk = raw[bps * pos:bps * (pos + pairs)]
        got, want = conv.convert(chunk), ref.convert(chunk)
        assert got.size == want.size == 2 * pairs
        assert np.array_equal(got, want), (pairs, np.nonzero(got != want)[0][:4])
        pos += pairs
    assert conv.mismatches() == 0                         # every speculative segment start was right


def test_airspy_late_merging_segments_are_repaired(gpu):
    """A slow, noiseless square wave: on its flat stretches the float recursion stalls next to its fixed point and the
    guessed and true averages of whole runs of segments never become bit-identical.  The repair walk redoes each run
    from the true value in front of it (runs in parallel); the result must be the Java's and the sequential fallback
    must not be needed."""
    from sdrtrunk_b200.dsp import AirspySampleConverter
    n = 40 * 2048
    t = np.arange(n)
    x = 300.0 / 2048 * np.sign(np.sin(t * 0.001)) + 5.0 / 2048
    for packed in (False, True):
        raw = sg.airspy_raw(x, packed)
        ref, conv = oracle.AirspySampleConverter(), AirspySampleConverter(maxSamples=1 << 17)
        ref.setSamplePacking(packed)
        conv.setSamplePacking(packed)
        for _ in range(3):
            assert np.array_equal(conv.convert(raw), ref.convert(raw))
        assert conv.mismatches() == 0
        assert conv.repaired() > 0


@pytest.mark.parametrize("walk", [True, False])
def test_airspy_speculation_fallback_is_exact(gpu, monkeypatch, walk):
    """A pathological stream defeats the speculation altogether: with constant samples the recursion stalls half an ulp
    short of its fixed point, on the side it came from.  The true average comes down from 0.9 and stalls just above
    0.75; the guesses stall elsewhere, segments agree and disagree with their neighbours at random and no repair walk
    starts from a true value except the first, which runs into the next one.  The verification must notice (every start
    against its predecessor's end) and the sequential fallback of the commit step must still give the Java's result --
    with the repair walk and without it (SDRGPU_AIRSPY_WALK=0)."""
    from sdrtrunk_b200.dsp import AirspySampleConverter
    if not walk:
        monkeypatch.setenv("SDRGPU_AIRSPY_WALK", "0")
    n = 4 * 4096 + 512
    ref, conv = oracle.AirspySampleConverter(), AirspySampleConverter(maxSamples=1 << 16)
    monkeypatch.delenv("SDRGPU_AIRSPY_WALK", raising=False)
    high, flat = sg.airspy_raw(np.full(n, 0.9)), sg.airspy_raw(np.full(n, 0.75))
    assert np.array_equal(conv.convert(high), ref.convert(high))
    for _ in range(3):
        assert np.array_equal(conv.convert(flat), ref.convert(flat))
    assert conv.mismatches() > 0


def test_channelizer_takes_airspy_buffers(gpu):
    """sdrgpu_chan_set_input_format(AIRSPY_*): raw buffers in, channels out = converter followed by the channelizer"""
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    m = 400
    rng = np.random.default_rng(9)
    n_complex = 40 * (m // 2)
    x = sg.airspy_real_signal(rng, 2 * n_complex, [(25000.0 * 7 + 3000, 0.2), (-25000.0 * 30 - 1000, 0.1)], fs=20e6)
    taps = oracle.sinc_m2_channelizer(25000.0, m, 9)
    for packed in (False, True):
        raw = sg.airspy_raw(x, packed)
        ref = oracle.AirspySampleConverter()
        ref.setSamplePacking(packed)
        iq = ref.convert(raw)
        plain = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
        want = np.concatenate([plain.receive(iq[:2 * 3000]), plain.receive(iq[2 * 3000:])])
        ch = ComplexPolyphaseChannelizerM2(taps, 25000 * m, m)
        ch.setSampleFormat("airspy_packed" if packed else "airspy")
        values = raw if packed else raw.view("<u2")
        cut = 3000 * (3 if packed else 2)                 # 3000 complex samples
        got = np.concatenate([ch.receive(values[:cut]), ch.receive(values[cut:])])
        assert np.array_equal(got, want)
