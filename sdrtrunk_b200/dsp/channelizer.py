"""Polyphase channelizer host mirror.

ComplexPolyphaseChannelizerM2 (J/dsp/filter/channelizer/ComplexPolyphaseChannelizerM2.java:64-449),
ChannelCalculator (.../ChannelCalculator.java:27-558) and TunerChannel (J/source/tuner/channel/TunerChannel.java)
with the reference's constructor / method names.  `float[]` buffers are numpy float32 arrays (interleaved
I,Q); device-resident callers pass integer device addresses instead.
"""
import ctypes as C

import numpy as np

from .. import native
from .filter_factory import FilterFactory


class TunerChannel:
    """J/source/tuner/channel/TunerChannel.java: centre frequency (Hz) + bandwidth (Hz)."""

    def __init__(self, frequency, bandwidth):
        self.mFrequency = int(frequency)
        self.mBandwidth = int(bandwidth)

    def getFrequency(self):
        return self.mFrequency

    def getBandwidth(self):
        return self.mBandwidth

    def getMinFrequency(self):
        return self.mFrequency - (self.mBandwidth // 2)

    def getMaxFrequency(self):
        return self.mFrequency + (self.mBandwidth // 2)


class ChannelCalculator:
    """ChannelCalculator.java: maps a TunerChannel to 1 or 2 polyphase bin indexes."""

    def __init__(self, sampleRate, channelCount, centerFrequency, oversampling=2.0):
        self.mSampleRate = float(sampleRate)
        self.mChannelCount = int(channelCount)
        self.mCenterFrequency = float(centerFrequency)
        self.mOversampling = float(oversampling)

    def getChannelBandwidth(self):
        return self.mSampleRate / self.mChannelCount

    def getChannelSampleRate(self):
        return self.getChannelBandwidth() * self.mOversampling

    def getChannelCount(self):
        return self.mChannelCount

    def getWrapAroundIndex(self):
        return self.mChannelCount // 2

    def setCenterFrequency(self, frequency):
        self.mCenterFrequency = float(frequency)

    def setRates(self, sampleRate, channelCount):
        self.mSampleRate = float(sampleRate)
        self.mChannelCount = int(channelCount)

    def getChannelIndexes(self, tunerChannel):
        idx = (C.c_int * 64)()
        n = C.c_int(0)
        native.check(native.lib().sdrgpu_channel_indexes(
            self.mSampleRate, self.mChannelCount, self.mCenterFrequency, tunerChannel.getFrequency(),
            tunerChannel.getBandwidth(), idx, 64, C.byref(n)))
        return list(idx[:n.value])

    def getCenterFrequencyForIndexes(self, indexes):
        if len(indexes) == 0:
            raise native.IllegalArgumentException("Indexes cannot be empty")
        arr = (C.c_int * len(indexes))(*indexes)
        f = C.c_longlong(0)
        native.check(native.lib().sdrgpu_center_frequency_for_indexes(
            self.mSampleRate, self.mChannelCount, self.mCenterFrequency, arr, len(indexes), C.byref(f)))
        return f.value


class ComplexPolyphaseChannelizerM2:
    """GPU-backed ComplexPolyphaseChannelizerM2.

    Constructors (as the reference, :93-126):
        ComplexPolyphaseChannelizerM2(taps, sampleRate, channelCount)
        ComplexPolyphaseChannelizerM2(sampleRate, tapsPerChannel)      -- designs the prototype filter
    receive(samples) returns the ReusableChannelResultsBuffer content: one float[2*M] row per block after the
    inverse FFT; receiveChannels(samples) returns the selected channels' contiguous streams (the product of
    ReusableChannelResultsBuffer.getChannel + OneChannelOutputProcessor for every registered channel).
    """

    DEFAULT_MINIMUM_CHANNEL_BANDWIDTH = 25000

    def __init__(self, *args, device=0, maxInputFloats=1 << 21):
        native.init(device)
        if len(args) == 3:
            taps, sampleRate, channelCount = args
            taps = native.f32(taps)
            if int(channelCount) % 2 != 0:
                raise native.IllegalArgumentException(
                    "Channel count must be an even multiple of the over-sample rate (2x)")
        elif len(args) == 2:
            sampleRate, tapsPerChannel = args
            channelCount = self.getChannelCount(sampleRate)
            taps = FilterFactory.getSincM2Channelizer(float(sampleRate) / channelCount, channelCount,
                                                      int(tapsPerChannel), False)
        else:
            raise TypeError("ComplexPolyphaseChannelizerM2(taps, sampleRate, channelCount) or (sampleRate, tapsPerChannel)")
        self.mSampleRate = float(sampleRate)
        self.mChannelCount = int(channelCount)
        self.mTapsPerChannel = -(-taps.size // self.mChannelCount)
        self.mTaps = taps
        self._max_input_floats = int(maxInputFloats)
        self._h = C.c_void_p()
        native.check(native.lib().sdrgpu_chan_create(C.byref(self._h), taps.ctypes.data_as(C.POINTER(C.c_float)),
                                                     taps.size, self.mChannelCount, self._max_input_floats))
        native.check(native.lib().sdrgpu_chan_set_sample_rate(self._h, self.mSampleRate))
        self._n_selected = self.mChannelCount

    # ---- reference API
    @staticmethod
    def getChannelCount(sampleRate=None):
        return native.lib().sdrgpu_channel_count_for_rate(float(sampleRate))

    def getSubChannelCount(self):
        return 2 * self.mChannelCount

    def getSampleRate(self):
        return self.mSampleRate

    def getChannelSampleRate(self):
        return self.mSampleRate / self.mChannelCount * 2.0

    def start(self):
        pass

    def stop(self):
        native.check(native.lib().sdrgpu_chan_sync(self._h))

    def receive(self, samples, samples_mem=native.HOST, out=None, out_mem=native.HOST):
        """Channelizes one tuner buffer; returns float32 [n_blocks, 2*M] (FFT bin order, no gain)."""
        return self._process(samples, samples_mem, out, out_mem, native.LAYOUT_RESULTS)

    # ---- per-channel extraction (seam 2 of SURVEY.md section 8b)
    def setChannels(self, bins, gain=None):
        """Selects the polyphase bins to extract (one OneChannelOutputProcessor each, gain = channel count)."""
        gain = float(self.mChannelCount) if gain is None else float(gain)
        arr = (native.OutputChannel * len(bins))()
        for i, b in enumerate(bins):
            arr[i] = native.OutputChannel(int(b), -1, 0, gain)
        native.check(native.lib().sdrgpu_chan_select(self._h, arr, len(bins), None, 0))
        self._n_selected = len(bins)

    POLYPHASE_SYNTHESIZER_TAPS_PER_CHANNEL = 9   # PolyphaseChannelManager.java

    def setOutputChannels(self, channels, synthesisFilter=None):
        """General selection: `channels` is a list of (indexes, frequencyOffsetHz[, gain]) where indexes is the 1- or
        2-element list ChannelCalculator.getChannelIndexes returns (PolyphaseChannelManager.getOutputProcessor,
        :198-222: One/TwoChannelOutputProcessor, gain = channel count).  The two-channel synthesis filter defaults to
        getSincM2Synthesizer(channelSampleRate, channelBandwidth, 2, 9) (getOutputProcessorFilter, :491-504)."""
        arr, any_two = self._output_channels(channels)
        filt, n_filt = None, 0
        if any_two:
            if synthesisFilter is None:
                synthesisFilter = FilterFactory.getSincM2Synthesizer(self.getChannelSampleRate(),
                                                                     self.mSampleRate / self.mChannelCount, 2,
                                                                     self.POLYPHASE_SYNTHESIZER_TAPS_PER_CHANNEL)
            filt, n_filt = self._synthesis_filter(synthesisFilter)
        native.check(native.lib().sdrgpu_chan_select(self._h, arr, len(channels), filt, n_filt))
        self._n_selected = len(channels)

    def updateOutputChannels(self, channels, previous, synthesisFilter=None):
        """Edits the running selection without resetting the channels it keeps (sdrgpu_chan_update_selection):
        `channels` as for setOutputChannels, previous[i] the index in the current selection that entry i continues (its
        output processor carries on, as after setPolyphaseChannelIndices / setFrequencyOffset) or -1 for a new channel.
        Channels no entry continues are removed.  A kept entry keeps its bin count and gain.  synthesisFilter=None keeps
        the current two-bin synthesis filter.  Takes effect from the next call that runs this channelizer."""
        if len(previous) != len(channels):
            raise native.IllegalArgumentException("one previous index per channel")
        arr, _ = self._output_channels(channels)
        prev = (C.c_int * len(channels))(*[int(p) for p in previous])
        filt, n_filt = (None, 0) if synthesisFilter is None else self._synthesis_filter(synthesisFilter)
        native.check(native.lib().sdrgpu_chan_update_selection(self._h, arr, prev, len(channels), filt, n_filt))
        self._n_selected = len(channels)

    def _output_channels(self, channels):
        arr = (native.OutputChannel * len(channels))()
        any_two = False
        for i, ch in enumerate(channels):
            indexes, offset = ch[0], ch[1]
            gain = float(ch[2]) if len(ch) > 2 else float(self.mChannelCount)
            if len(indexes) not in (1, 2):
                raise native.IllegalArgumentException(
                    "Request to create an output processor for unexpected channel index size:%d" % len(indexes))
            any_two |= len(indexes) == 2
            arr[i] = native.OutputChannel(int(indexes[0]), int(indexes[1]) if len(indexes) == 2 else -1, int(offset), gain)
        return arr, any_two

    def _synthesis_filter(self, synthesisFilter):
        self._synth = native.f32(synthesisFilter)
        return self._synth.ctypes.data_as(C.POINTER(C.c_float)), self._synth.size

    def setFrequencyOffsets(self, offsets):
        """ChannelOutputProcessor.setFrequencyOffset for running channels: `offsets` maps an index into the current
        selection (setOutputChannels / setChannels order) to its new frequency offset in Hz.  Takes effect from the next
        call that runs this channelizer (receiveChannels or a pipeline call); only the oscillators' angles change, as in
        the reference, and every other channel is untouched (sdrgpu_chan_set_frequency_offsets)."""
        items = [(int(k), int(v)) for k, v in dict(offsets).items()]
        if not items:
            return
        idx = (C.c_int * len(items))(*[k for k, _ in items])
        hz = (C.c_longlong * len(items))(*[v for _, v in items])
        native.check(native.lib().sdrgpu_chan_set_frequency_offsets(self._h, idx, hz, len(items)))

    def setFrequencyOffset(self, index, frequencyOffset):
        """the one-channel form of setFrequencyOffsets"""
        self.setFrequencyOffsets({index: frequencyOffset})

    def receiveChannels(self, samples, samples_mem=native.HOST, out=None, out_mem=native.HOST, out_stride_floats=None):
        """Returns float32 [n_selected, 2*n_blocks]: each row one channel's interleaved I/Q stream."""
        return self._process(samples, samples_mem, out, out_mem, native.LAYOUT_CHANNELS, out_stride_floats)

    _FORMATS = {"f32": (native.FORMAT_F32, np.float32), "u8": (native.FORMAT_U8, np.uint8),
                "s8": (native.FORMAT_S8, np.int8), "s16le": (native.FORMAT_S16LE, np.dtype("<i2")),
                "airspy": (native.FORMAT_AIRSPY_U16LE, np.dtype("<u2")),
                "airspy_packed": (native.FORMAT_AIRSPY_PACKED12, np.uint8)}

    def setSampleFormat(self, fmt):
        """Native tuner sample format of the buffers given to receive / receiveChannels: 'f32' (default), 'u8'
        (ByteSampleConverter), 's8' (SignedByteSampleConverter), 's16le' (ConversionUtils), 'airspy' / 'airspy_packed'
        (AirspySampleConverter: 12-bit real samples, two per complex sample; uint16 values or packed bytes);
        converted on the device."""
        code, self._dtype = self._FORMATS[fmt]
        self._packed = fmt == "airspy_packed"
        native.check(native.lib().sdrgpu_chan_set_input_format(self._h, code))

    def setStream(self, cuda_stream):
        native.check(native.lib().sdrgpu_chan_set_stream(self._h, C.c_void_p(int(cuda_stream) if cuda_stream else 0)))

    def sync(self):
        native.check(native.lib().sdrgpu_chan_sync(self._h))

    def enableTiming(self, on=True):
        native.check(native.lib().sdrgpu_chan_enable_timing(self._h, 1 if on else 0))

    def lastKernelMs(self):
        ms = C.c_float(0)
        native.check(native.lib().sdrgpu_chan_last_kernel_ms(self._h, C.byref(ms)))
        return ms.value

    def blocksFor(self, n_floats):
        return native.lib().sdrgpu_chan_blocks_for(self._h, int(n_floats))

    def _process(self, samples, samples_mem, out, out_mem, layout, out_stride_floats=None):
        L = native.lib()
        if samples_mem == native.HOST:
            samples = np.ascontiguousarray(samples, dtype=getattr(self, "_dtype", np.float32))
            n_floats = samples.size // 3 * 2 if getattr(self, "_packed", False) else samples.size
            in_ptr = native.ptr(samples)
        else:
            in_ptr, n_floats = native.ptr(samples[0]), int(samples[1])
        n_blocks = L.sdrgpu_chan_blocks_for(self._h, n_floats)
        rows = self._n_selected if layout == native.LAYOUT_CHANNELS else n_blocks
        cols = 2 * n_blocks if layout == native.LAYOUT_CHANNELS else 2 * self.mChannelCount
        if out_mem == native.HOST:
            if out is None:
                out = np.empty((rows, cols), np.float32)
            out_ptr = native.ptr(out)
            stride = cols
        else:
            out_ptr = native.ptr(out)
            stride = int(out_stride_floats) if out_stride_floats else cols
        got = C.c_int(0)
        native.check(L.sdrgpu_chan_process(self._h, in_ptr, n_floats, samples_mem, out_ptr, stride, out_mem, layout,
                                           C.byref(got)))
        assert got.value == n_blocks
        return out if out_mem == native.HOST else n_blocks

    def dispose(self):
        if getattr(self, "_h", None) is not None and self._h:
            native.lib().sdrgpu_chan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.dispose()
        except Exception:
            pass


class _SampleConverter:
    """NativeBufferConverter.convertSamples(ByteBuffer, length) -> float[]: converts on the device"""
    FORMAT, DTYPE = None, None

    def convertSamples(self, nativeBuffer, length=None):
        raw = np.ascontiguousarray(np.frombuffer(bytes(nativeBuffer), dtype=self.DTYPE))
        n = raw.size if length is None else min(raw.size, int(length) // raw.itemsize)
        out = np.empty(n, np.float32)
        native.init(0)
        native.check(native.lib().sdrgpu_convert_samples(self.FORMAT, native.ptr(raw), native.HOST, n, native.ptr(out),
                                                         native.HOST))
        return out


class AirspySampleConverter:
    """J/source/tuner/airspy/AirspySampleConverter.java: raw 12-bit real samples -> DC removal -> Hilbert transform ->
    interleaved I/Q, on the device (bit-exact; state carries from buffer to buffer as in the Java object)."""

    def __init__(self, maxSamples=1 << 20, device=0):
        native.init(device)
        self._h = C.c_void_p()
        self._max = int(maxSamples)
        self._packed = False
        native.check(native.lib().sdrgpu_airspy_create(C.byref(self._h), self._max))

    def setSamplePacking(self, enabled):
        self._packed = bool(enabled)
        native.check(native.lib().sdrgpu_airspy_set_sample_packing(self._h, 1 if enabled else 0))

    def convert(self, raw):
        """raw: the native buffer's bytes (uint8).  Returns float32 interleaved I/Q, one float per real sample."""
        raw = np.ascontiguousarray(raw, np.uint8)
        n = raw.size // 3 * 2 if self._packed else raw.size // 2
        out = np.empty(n, np.float32)
        native.check(native.lib().sdrgpu_airspy_convert(self._h, native.ptr(raw), native.HOST, n, native.ptr(out), native.HOST))
        return out

    def mismatches(self):
        """segments that forced a call onto the sequential fallback (see sdrgpu_airspy_mismatches)"""
        c = C.c_int(0)
        native.check(native.lib().sdrgpu_airspy_mismatches(self._h, C.byref(c)))
        return c.value

    def repaired(self):
        """segments redone in parallel because their speculative start had not merged (sdrgpu_airspy_repaired)"""
        c = C.c_int(0)
        native.check(native.lib().sdrgpu_airspy_repaired(self._h, C.byref(c)))
        return c.value

    def dispose(self):
        if getattr(self, "_h", None) is not None and self._h:
            native.lib().sdrgpu_airspy_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.dispose()
        except Exception:
            pass


class ByteSampleConverter(_SampleConverter):
    """J/source/tuner/usb/converter/ByteSampleConverter.java"""
    FORMAT, DTYPE = native.FORMAT_U8, np.uint8


class SignedByteSampleConverter(_SampleConverter):
    """J/source/tuner/usb/converter/SignedByteSampleConverter.java"""
    FORMAT, DTYPE = native.FORMAT_S8, np.int8


class Signed16BitSampleConverter(_SampleConverter):
    """J/sample/ConversionUtils.java:22-34 convertFromSigned16BitSamples"""
    FORMAT, DTYPE = native.FORMAT_S16LE, np.dtype("<i2")
