"""Per-channel banks: host mirror of the reference's per-channel DSP classes on top of sdrgpu_bank.

`Bank` is the many-channel primitive (C independent channel streams through one chain).  The classes below it
keep the reference's names and method signatures for a single channel (the drop-in shape), each backed by a
one-channel bank:

    ComplexFIRFilter2 / RealFIRFilter2          J/dsp/filter/fir/complex/ComplexFIRFilter2.java, real/RealFIRFilter2.java
    DecimationFilterFactory + decimation filters J/dsp/filter/decimate/DecimationFilterFactory.java:36-104
    ComplexFeedForwardGainControl               J/dsp/gain/ComplexFeedForwardGainControl.java:147-181
    FMDemodulator / SquelchingFMDemodulator      J/dsp/fm/FMDemodulator.java, SquelchingFMDemodulator.java
    CostasLoop, PLLBandwidth, InterpolatingSampleBuffer, DQPSKDecisionDirectedDemodulator,
    DQPSKGardnerDemodulator                     J/dsp/psk/..., J/dsp/psk/pll/...
"""
import ctypes as C
import enum

import numpy as np

from .. import native


class Dibit(enum.Enum):
    """J/dsp/symbol/Dibit.java:27-30 (getValue)"""
    D00_PLUS_1 = 0
    D01_PLUS_3 = 1
    D10_MINUS_1 = 2
    D11_MINUS_3 = 3

    def getValue(self):
        return self.value


class PLLBandwidth(enum.Enum):
    """J/dsp/psk/pll/PLLBandwidth.java:34-37"""
    BW_400 = 400.0
    BW_300 = 300.0
    BW_250 = 250.0
    BW_200 = 200.0

    def getLoopBandwidth(self):
        return self.value


class Bank:
    """C independent channel streams through [decimate] -> [FIR] -> [AGC] -> demodulator on the GPU."""

    def __init__(self, n_channels, sample_rate, demod=native.DEMOD_NONE, fir_taps=None, fir_gain=1.0, agc=False,
                 decimation=0, block_size=1024, symbol_rate=0.0, pll_bandwidth=0.0, sample_counter_gain=0.0,
                 fm_gain=1.0, squelch_alpha=0.0004, squelch_threshold_db=-78.0, squelch_ramp=4,
                 max_samples_per_call=1 << 16, device=0):
        native.init(device)
        self.n_channels = int(n_channels)
        self.sample_rate = float(sample_rate)
        self.demod = demod
        self.decimation = int(decimation)
        self.block_size = int(block_size)
        self._taps = native.f32(fir_taps) if fir_taps is not None and len(fir_taps) else None
        cfg = native.BankConfig()
        cfg.n_channels = self.n_channels
        cfg.sample_rate = self.sample_rate
        cfg.decimation = self.decimation
        cfg.fir_taps = self._taps.ctypes.data_as(C.POINTER(C.c_float)) if self._taps is not None else None
        cfg.n_fir_taps = self._taps.size if self._taps is not None else 0
        cfg.fir_gain = float(fir_gain)
        cfg.agc = 1 if agc else 0
        cfg.block_size = self.block_size
        cfg.demod = demod
        cfg.symbol_rate = float(symbol_rate)
        cfg.pll_bandwidth = float(pll_bandwidth)
        cfg.sample_counter_gain = float(sample_counter_gain)
        cfg.fm_gain = float(fm_gain)
        cfg.squelch_alpha = float(squelch_alpha)
        cfg.squelch_threshold_db = float(squelch_threshold_db)
        cfg.squelch_ramp = int(squelch_ramp)
        cfg.max_samples_per_call = int(max_samples_per_call)
        self.max_samples_per_call = int(max_samples_per_call)
        self._h = C.c_void_p()
        native.check(native.lib().sdrgpu_bank_create(C.byref(self._h), C.byref(cfg)))
        self._pending = 0

    @classmethod
    def preset(cls, preset, n_channels, sample_rate, fir_taps=None, max_samples_per_call=1 << 16, device=0):
        """Decoder front-end presets (P25P1DecoderC4FM / LSM / P25P2DecoderHDQPSK / NBFMDecoder constants)."""
        native.init(device)
        taps = native.f32(fir_taps) if fir_taps is not None else None
        cfg = native.BankConfig()
        native.check(native.lib().sdrgpu_bank_config_preset(
            C.byref(cfg), preset, int(n_channels), float(sample_rate),
            taps.ctypes.data_as(C.POINTER(C.c_float)) if taps is not None else None,
            taps.size if taps is not None else 0, int(max_samples_per_call)))
        return cls(cfg.n_channels, cfg.sample_rate, cfg.demod, taps if cfg.n_fir_taps else None, cfg.fir_gain,
                   bool(cfg.agc), cfg.decimation, cfg.block_size, cfg.symbol_rate, cfg.pll_bandwidth,
                   cfg.sample_counter_gain, cfg.fm_gain, cfg.squelch_alpha, cfg.squelch_threshold_db,
                   cfg.squelch_ramp, max_samples_per_call, device)

    # ---- sizes
    @property
    def is_dqpsk(self):
        return self.demod in (native.DEMOD_DQPSK_DECISION, native.DEMOD_DQPSK_GARDNER)

    @property
    def is_fm(self):
        return self.demod in (native.DEMOD_FM, native.DEMOD_FM_SQUELCH)

    def _outputs_for(self, n_samples):
        blocks = (self._pending + n_samples) // self.block_size
        per_block = self.block_size // max(self.decimation, 1)
        return blocks, blocks * per_block

    def process(self, iq, want_filtered=False, want_squelch=False):
        """iq: float32 [C, 2*n] (interleaved I/Q per channel row).  Returns
        DQPSK: list of uint8 dibit arrays per channel (and the AGC output [C, 2*n_out] if want_filtered)
        FM:    float32 [C, n_out] demodulated samples;  NONE: float32 [C, 2*n_out] filtered complex stream.
        want_squelch (FM_SQUELCH banks): also uint8 [C, buffers] squelch statuses, one per assembler buffer consumed
        (native.SQUELCH_ATTACK .. _UNMUTE | native.SQUELCH_CHANGED), i.e. (demodulated, statuses)."""
        iq = native.f32(iq)
        if iq.ndim == 1:
            iq = iq.reshape(1, -1)
        assert iq.shape[0] == self.n_channels and iq.shape[1] % 2 == 0
        n = iq.shape[1] // 2
        blocks, n_out = self._outputs_for(n)
        status = self._status_rows(blocks) if want_squelch else None
        self._pending = (self._pending + n) % self.block_size
        counts = np.zeros(self.n_channels, np.int32)
        L = native.lib()
        if self.is_dqpsk:
            stride = max(16, n_out // 3 + 16)
            symbols = np.zeros((self.n_channels, stride), np.uint8)
            filt = np.zeros((self.n_channels, max(2 * n_out, 2)), np.float32) if want_filtered else None
            native.check(L.sdrgpu_bank_process(self._h, native.ptr(iq), iq.shape[1], n, native.HOST, native.ptr(symbols),
                                               stride, native.ptr(filt) if want_filtered else None,
                                               filt.shape[1] if want_filtered else 0, native.ptr(counts), native.HOST))
            out = [symbols[c, :counts[c]].copy() for c in range(self.n_channels)]
            return (out, filt[:, :2 * n_out]) if want_filtered else out
        width = n_out if self.is_fm else 2 * n_out
        dem = np.zeros((self.n_channels, max(width, 1)), np.float32)
        native.check(L.sdrgpu_bank_process(self._h, native.ptr(iq), iq.shape[1], n, native.HOST, native.ptr(status),
                                           status.shape[1] if status is not None else 0, native.ptr(dem), dem.shape[1],
                                           native.ptr(counts), native.HOST))
        if status is not None:
            return dem[:, :width], status[:, :blocks]
        return dem[:, :width]

    def _status_rows(self, blocks):
        """host rows for the squelch statuses of a call that consumes `blocks` buffers (turns the bank's status
        reporting on)"""
        if self.demod != native.DEMOD_FM_SQUELCH:
            raise native.IllegalArgumentException("squelch statuses come from SquelchingFMDemodulator banks only")
        if not getattr(self, "_reporting", False):
            native.check(native.lib().sdrgpu_bank_set_squelch_reporting(self._h, 1))
            self._reporting = True
        return np.zeros((self.n_channels, max(blocks, 1)), np.uint8)

    def setSquelchThreshold(self, threshold_db, channel=-1):
        """PowerSquelch.setSquelchThreshold (dB) of one channel, or of every channel (channel = -1), from the next
        buffer on; the squelch's IIR and ramp state carry on"""
        native.check(native.lib().sdrgpu_bank_set_squelch_threshold(self._h, int(channel), float(threshold_db)))

    def correctInversion(self, channel, radians):
        native.check(native.lib().sdrgpu_bank_correct_inversion(self._h, int(channel), float(radians)))

    def setSyncDetector(self, kind):
        """P25P1SyncDetector / P25P2SyncDetector + PLLPhaseInversionDetector feedback on the device
        (native.SYNC_P25_PHASE1 / SYNC_P25_PHASE2 / SYNC_NONE).  Symbol bytes become dibit | event << 2 | errors << 5."""
        native.check(native.lib().sdrgpu_bank_set_sync_detector(self._h, int(kind)))

    def setDemodulatorLanes(self, lanes):
        """tuning / testing: 32, 16, 8, 4 or 1 lanes of a warp per channel in the demodulator kernel, 0 = automatic"""
        native.check(native.lib().sdrgpu_bank_set_demodulator_lanes(self._h, int(lanes)))

    def resetPLL(self, channel):
        native.check(native.lib().sdrgpu_bank_reset_pll(self._h, int(channel)))

    def setSymbolTap(self, channel):
        """Per-symbol tap points of one channel (the listeners of DQPSKDecisionDirectedDemodulatorInstrumented /
        DQPSKGardnerDemodulatorInstrumented: setComplexSymbolListener, setSamplesPerSymbolListener, setPLLErrorListener,
        setPLLFrequencyListener); None / -1 clears it."""
        native.check(native.lib().sdrgpu_bank_set_symbol_tap(self._h, -1 if channel is None else int(channel)))

    def symbolTap(self, sampleRate=None):
        """float64 [n_symbols, 6] of the last process call: symbol I, symbol Q, detected samples per symbol, PLL frequency
        (radians per sample; in Hz when sampleRate is given, as the Java's listener reports it), sampling point, PLL error"""
        cap = 1 << 16
        out = np.zeros((cap, 6), np.float64)
        n = C.c_int(0)
        native.check(native.lib().sdrgpu_bank_read_symbol_tap(self._h, out.ctypes.data_as(C.POINTER(C.c_double)), cap, C.byref(n)))
        out = out[:n.value].copy()
        if sampleRate is not None:
            out[:, 3] *= float(sampleRate) / (2.0 * np.pi)
        return out

    def loopState(self, channel):
        st = (C.c_double * 4)()
        native.check(native.lib().sdrgpu_bank_get_loop_state(self._h, int(channel), st))
        return tuple(st)

    def setStream(self, cuda_stream):
        native.check(native.lib().sdrgpu_bank_set_stream(self._h, C.c_void_p(int(cuda_stream) if cuda_stream else 0)))

    def sync(self):
        native.check(native.lib().sdrgpu_bank_sync(self._h))

    def enableTiming(self, on=True):
        native.check(native.lib().sdrgpu_bank_enable_timing(self._h, 1 if on else 0))

    def lastKernelMs(self):
        ms = (C.c_float * 2)()
        native.check(native.lib().sdrgpu_bank_last_kernel_ms(self._h, ms))
        return ms[0], ms[1]

    def dispose(self):
        if getattr(self, "_h", None) is not None and self._h:
            native.lib().sdrgpu_bank_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.dispose()
        except Exception:
            pass


class Pipeline:
    """channelizer(s) -> bank on the device (sdrgpu_pipeline): only dibits / demodulated floats come back.

    `channelizer` may be a list of channelizers of equal channel count (several tuners): their selected channels are
    consecutive row ranges of the one bank, and process() then takes one sample buffer per tuner
    (sdrgpu_pipeline_create_multi: the reference runs every channel as its own task whichever tuner it came from,
    J/source/tuner/channel/TunerChannelSource.java:290-319).

    Pipeline(channelizers, banks=[...], route=[...]) feeds several banks (decoder types) from the same channelizer pass
    (sdrgpu_pipeline_create_routed): route[r] is the index in `banks` of the bank that decodes selected channel r, in
    pipeline row order (the first channelizer's selection, then the next one's, ...), and process() returns one list of
    per-row results per bank."""

    def __init__(self, channelizer, bank=None, banks=None, route=None):
        self.channelizers = list(channelizer) if isinstance(channelizer, (list, tuple)) else [channelizer]
        self.channelizer = self.channelizers[0]
        self.routed = banks is not None
        self.banks = list(banks) if self.routed else [bank]
        self.bank = self.banks[0]
        self._h = C.c_void_p()
        handles = (C.c_void_p * len(self.channelizers))(*[c._h for c in self.channelizers])
        if self.routed:
            bank_handles = (C.c_void_p * len(self.banks))(*[b._h for b in self.banks])
            r = np.ascontiguousarray(route, dtype=np.int32)
            native.check(native.lib().sdrgpu_pipeline_create_routed(C.byref(self._h), handles, len(self.channelizers),
                                                                   bank_handles, len(self.banks),
                                                                   r.ctypes.data_as(C.POINTER(C.c_int))))
        else:
            native.check(native.lib().sdrgpu_pipeline_create_multi(C.byref(self._h), handles, len(self.channelizers), bank._h))
        self._pending = 0

    def setChunks(self, chunks):
        native.check(native.lib().sdrgpu_pipeline_set_chunks(self._h, int(chunks)))

    def setDeviceChunks(self, chunks):
        native.check(native.lib().sdrgpu_pipeline_set_device_chunks(self._h, int(chunks)))

    def process(self, samples, samples_mem=native.HOST, n_floats=None, want_squelch=False):
        """samples: interleaved tuner I/Q in the channelizer's input format (one array, or one per tuner).  Returns
        per-channel dibit arrays (DQPSK) or demod floats, indexed by bank row.  want_squelch: every FM_SQUELCH bank's
        result is (demodulated, squelch statuses), as Bank.process gives them."""
        L = native.lib()
        bank = self.bank
        multi = len(self.channelizers) > 1
        bufs = list(samples) if multi else [samples]
        assert len(bufs) == len(self.channelizers)
        if samples_mem == native.HOST:
            bufs = [np.ascontiguousarray(b, dtype=getattr(self.channelizer, "_dtype", np.float32)) for b in bufs]
            n_floats = bufs[0].size // 3 * 2 if getattr(self.channelizer, "_packed", False) else bufs[0].size
            assert all(b.size == bufs[0].size for b in bufs)
        else:
            n_floats = int(n_floats)
        in_ptrs = (C.c_void_p * len(bufs))(*[C.cast(native.ptr(b), C.c_void_p) for b in bufs])
        n = self.channelizer.blocksFor(n_floats)
        blocks = (self._pending + n) // bank.block_size
        n_out = blocks * (bank.block_size // max(bank.decimation, 1))
        self._pending = (self._pending + n) % bank.block_size
        if self.routed:
            return self._process_routed(in_ptrs, n_floats, samples_mem, blocks, want_squelch)
        counts = np.zeros(bank.n_channels, np.int32)
        if bank.is_dqpsk:
            stride = max(16, n_out // 3 + 16)
            symbols = np.zeros((bank.n_channels, stride), np.uint8)
            native.check(L.sdrgpu_pipeline_process_multi(self._h, in_ptrs, n_floats, samples_mem, native.ptr(symbols), stride,
                                                         None, 0, native.ptr(counts), native.HOST))
            return [symbols[c, :counts[c]].copy() for c in range(bank.n_channels)]
        width = n_out if bank.is_fm else 2 * n_out
        dem = np.zeros((bank.n_channels, max(width, 1)), np.float32)
        status = bank._status_rows(blocks) if want_squelch else None
        native.check(L.sdrgpu_pipeline_process_multi(self._h, in_ptrs, n_floats, samples_mem, native.ptr(status),
                                                     status.shape[1] if status is not None else 0, native.ptr(dem),
                                                     dem.shape[1], native.ptr(counts), native.HOST))
        if status is not None:
            return dem[:, :width], status[:, :blocks]
        return dem[:, :width]

    def _process_routed(self, in_ptrs, n_floats, samples_mem, blocks, want_squelch=False):
        """every bank's outputs in the shape Pipeline.process gives for one bank: dibit arrays per row (DQPSK), else
        demodulated floats [rows, n]"""
        outs = (native.BankOutput * len(self.banks))()
        keep = []
        for o, bank in zip(outs, self.banks):
            n_out = blocks * (bank.block_size // max(bank.decimation, 1))
            counts = np.zeros(bank.n_channels, np.int32)
            o.counts = counts.ctypes.data
            if bank.is_dqpsk:
                stride = max(16, n_out // 3 + 16)
                buf = np.zeros((bank.n_channels, stride), np.uint8)
                o.symbols, o.symbol_stride = buf.ctypes.data, stride
            else:
                width = n_out if bank.is_fm else 2 * n_out
                buf = np.zeros((bank.n_channels, max(width, 1)), np.float32)
                o.demod, o.demod_stride_floats = buf.ctypes.data, buf.shape[1]
            status = None
            if want_squelch and bank.demod == native.DEMOD_FM_SQUELCH:
                status = bank._status_rows(blocks)
                o.symbols, o.symbol_stride = status.ctypes.data, status.shape[1]
            keep.append((bank, buf, counts, n_out, status))
        native.check(native.lib().sdrgpu_pipeline_process_routed(self._h, in_ptrs, n_floats, samples_mem, outs, native.HOST))
        result = []
        for bank, buf, counts, n_out, status in keep:
            if bank.is_dqpsk:
                result.append([buf[c, :counts[c]].copy() for c in range(bank.n_channels)])
            else:
                dem = buf[:, :n_out if bank.is_fm else 2 * n_out]
                result.append((dem, status[:, :blocks]) if status is not None else dem)
        return result

    def submit(self, samples):
        """asynchronous process() for a continuous stream of host buffers (DQPSK banks): enqueues the call and returns;
        wait() then returns the per-channel dibit arrays of the OLDEST call in flight.  At most two calls in flight
        (sdrgpu_pipeline_submit_multi / sdrgpu_pipeline_wait); the buffers are kept alive here until their wait()."""
        L = native.lib()
        bank = self.bank
        assert bank.is_dqpsk
        multi = len(self.channelizers) > 1
        bufs = list(samples) if multi else [samples]
        assert len(bufs) == len(self.channelizers)
        bufs = [np.ascontiguousarray(b, dtype=getattr(self.channelizer, "_dtype", np.float32)) for b in bufs]
        n_floats = bufs[0].size // 3 * 2 if getattr(self.channelizer, "_packed", False) else bufs[0].size
        assert all(b.size == bufs[0].size for b in bufs)
        in_ptrs = (C.c_void_p * len(bufs))(*[C.cast(native.ptr(b), C.c_void_p) for b in bufs])
        n = self.channelizer.blocksFor(n_floats)
        blocks = (self._pending + n) // bank.block_size
        n_out = blocks * (bank.block_size // max(bank.decimation, 1))
        stride = max(16, n_out // 3 + 16)
        symbols = np.zeros((bank.n_channels, stride), np.uint8)
        counts = np.zeros(bank.n_channels, np.int32)
        native.check(L.sdrgpu_pipeline_submit_multi(self._h, in_ptrs, n_floats, native.ptr(symbols), stride, native.ptr(counts)))
        self._pending = (self._pending + n) % bank.block_size
        if not hasattr(self, "_in_flight"):
            self._in_flight = []
        self._in_flight.append((bufs, in_ptrs, symbols, counts))

    def wait(self):
        """results of the oldest submitted call (None if nothing is in flight)"""
        if not getattr(self, "_in_flight", None):
            return None
        native.check(native.lib().sdrgpu_pipeline_wait(self._h))
        _, _, symbols, counts = self._in_flight.pop(0)
        return [symbols[c, :counts[c]].copy() for c in range(self.bank.n_channels)]

    def dispose(self):
        if getattr(self, "_h", None) is not None and self._h:
            native.lib().sdrgpu_pipeline_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.dispose()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------------------
# single-channel drop-in shapes
# ------------------------------------------------------------------------------------------------------------
class _LazyBank:
    """creates its one-channel bank at the first buffer (block size = that buffer's length, like the reference's
    fixed-size assembler buffers); later buffers must have the same length"""

    def __init__(self, **kw):
        self._kw = kw
        self._bank = None
        self._length = None

    def _get(self, n_samples):
        if self._bank is None:
            self._length = n_samples
            self._bank = Bank(1, block_size=n_samples, max_samples_per_call=n_samples, **self._kw)
        elif n_samples != self._length:
            raise native.IllegalArgumentException(
                "buffer length changed from %d to %d samples; GPU-backed filters need fixed-size buffers" %
                (self._length, n_samples))
        return self._bank


class ComplexFIRFilter2(_LazyBank):
    """ComplexFIRFilter2(float[] coefficients[, float gain]).filter(buffer)"""

    def __init__(self, coefficients, gain=1.0, sampleRate=50000.0):
        super().__init__(sample_rate=sampleRate, fir_taps=coefficients, fir_gain=gain)

    def filter(self, samples):
        samples = native.f32(samples)
        return self._get(samples.size // 2).process(samples.reshape(1, -1))[0]


class RealFIRFilter2(_LazyBank):
    """RealFIRFilter2(float[] coefficients[, float gain]).filter(float[]): the real stream rides the I rail"""

    def __init__(self, coefficients, gain=1.0, sampleRate=50000.0):
        super().__init__(sample_rate=sampleRate, fir_taps=coefficients, fir_gain=gain)

    def filter(self, samples):
        samples = native.f32(samples)
        iq = np.zeros(2 * samples.size, np.float32)
        iq[0::2] = samples
        return self._get(samples.size).process(iq.reshape(1, -1))[0][0::2].copy()


class ComplexFeedForwardGainControl(_LazyBank):
    """ComplexFeedForwardGainControl(window).filter(buffer): block AGC (the window argument is unused on this path)"""

    def __init__(self, window=32, sampleRate=50000.0):
        super().__init__(sample_rate=sampleRate, agc=True)

    def filter(self, samples):
        samples = native.f32(samples)
        return self._get(samples.size // 2).process(samples.reshape(1, -1))[0]


class _ComplexDecimationFilter(_LazyBank):
    def __init__(self, rate, sampleRate=50000.0):
        self.rate = rate
        super().__init__(sample_rate=sampleRate, decimation=rate)

    def decimateComplex(self, samples):
        samples = native.f32(samples)
        if self.rate and samples.size % (2 * self.rate) != 0:
            raise native.IllegalArgumentException(
                "Sample buffer length [%d] must be an integer multiple of %d" % (samples.size, 2 * self.rate))
        return self._get(samples.size // 2).process(samples.reshape(1, -1))[0]

    decimate = decimateComplex


class _RealDecimationFilter(_LazyBank):
    """IRealDecimationFilter.decimateReal(float[]): the real stream rides the I rail of the complex cascade (the
    half-band arithmetic is per rail, RealHalfBandDecimationFilter.java:61-111 == the complex one with Q absent)"""

    def __init__(self, rate, sampleRate=50000.0):
        self.rate = rate
        super().__init__(sample_rate=sampleRate, decimation=rate)

    def decimateReal(self, samples):
        samples = native.f32(samples)
        if self.rate and samples.size % self.rate != 0:
            raise native.IllegalArgumentException(
                "Sample buffer length [%d] must be an integer multiple of %d" % (samples.size, self.rate))
        iq = np.zeros(2 * samples.size, np.float32)
        iq[0::2] = samples
        return self._get(samples.size).process(iq.reshape(1, -1))[0][0::2].copy()


class DecimationFilterFactory:
    SUPPORTED_RATES = (0, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024)

    @staticmethod
    def getComplexDecimationFilter(decimationRate):
        if decimationRate not in DecimationFilterFactory.SUPPORTED_RATES:
            raise native.IllegalArgumentException("Unsupported decimation rate: %d.  Supported decimation rates are:%s" %
                                                  (decimationRate, DecimationFilterFactory.SUPPORTED_RATES))
        return _ComplexDecimationFilter(decimationRate)

    @staticmethod
    def getRealDecimationFilter(decimationRate):
        if decimationRate not in DecimationFilterFactory.SUPPORTED_RATES:
            raise native.IllegalArgumentException("Unsupported decimation rate: %d.  Supported decimation rates are:%s" %
                                                  (decimationRate, DecimationFilterFactory.SUPPORTED_RATES))
        return _RealDecimationFilter(decimationRate)


class FMDemodulator(_LazyBank):
    """FMDemodulator(float gain).demodulate(buffer) -> float[]"""

    def __init__(self, gain=1.0, sampleRate=25000.0):
        self.mGain = gain
        super().__init__(sample_rate=sampleRate, demod=native.DEMOD_FM, fm_gain=gain)

    def demodulate(self, samples):
        samples = native.f32(samples)
        return self._get(samples.size // 2).process(samples.reshape(1, -1))[0]


class SquelchingFMDemodulator(_LazyBank):
    """SquelchingFMDemodulator(alpha, threshold, ramp).demodulate(buffer) -> float[], and the squelch questions
    NBFMDecoder asks after each buffer: isSquelchChanged(), isMuted(), setSquelchThreshold(db)."""

    def __init__(self, alpha, threshold, ramp, sampleRate=25000.0):
        super().__init__(sample_rate=sampleRate, demod=native.DEMOD_FM_SQUELCH, squelch_alpha=alpha,
                         squelch_threshold_db=threshold, squelch_ramp=ramp)
        self._status = native.SQUELCH_MUTE      # PowerSquelch starts muted

    def demodulate(self, samples):
        samples = native.f32(samples)
        dem, status = self._get(samples.size // 2).process(samples.reshape(1, -1), want_squelch=True)
        self._status = int(status[0, -1])
        return dem[0]

    def isSquelchChanged(self):
        """the squelch changed state at least once during the last demodulate(buffer)"""
        return bool(self._status & native.SQUELCH_CHANGED)

    def isMuted(self):
        """passing no audio after the last buffer: the squelch is in MUTE or ATTACK, the states in which demodulate
        writes 0.0f (the reference's class has no such query; NBFMDecoder's use of the squelch state means this)"""
        return (self._status & 3) in (native.SQUELCH_MUTE, native.SQUELCH_ATTACK)

    def setSquelchThreshold(self, threshold):
        """PowerSquelch.setSquelchThreshold(dB): used from the next buffer on"""
        if self._bank is None:
            self._kw["squelch_threshold_db"] = float(threshold)
        else:
            self._bank.setSquelchThreshold(threshold)


class CostasLoop:
    """CostasLoop(sampleRate, symbolRate): the loop itself runs inside the demodulator kernel; this object carries
    its parameters and forwards correctInversion / reset to the device state."""

    def __init__(self, sampleRate, symbolRate):
        self.mSampleRate, self.mSymbolRate = float(sampleRate), float(symbolRate)
        self.mPLLBandwidth = PLLBandwidth.BW_400
        self._demod = None

    def setPLLBandwidth(self, pllBandwidth):
        if self._demod is not None and self._demod._bank is not None:
            raise native.IllegalStateException("PLL bandwidth must be set before the first buffer")
        self.mPLLBandwidth = pllBandwidth

    def correctInversion(self, correction):
        if self._demod is not None and self._demod._bank is not None:
            self._demod._bank.correctInversion(0, correction)

    def reset(self):
        if self._demod is not None and self._demod._bank is not None:
            self._demod._bank.resetPLL(0)

    def getLoopFrequency(self):
        return self._demod._bank.loopState(0)[1]


class InterpolatingSampleBuffer:
    """InterpolatingSampleBuffer(samplesPerSymbol, sampleCounterGain): parameters of the device-side buffer"""

    def __init__(self, samplesPerSymbol, sampleCounterGain):
        self.mSamplesPerSymbol = float(samplesPerSymbol)
        self.mSampleCounterGain = float(sampleCounterGain)


class _PSKDemodulator:
    KIND = None

    def __init__(self, phaseLockedLoop, interpolatingSampleBuffer):
        self.mPLL = phaseLockedLoop
        self.mBuffer = interpolatingSampleBuffer
        self.mSymbolListener = None
        self._bank = None
        self._length = None
        phaseLockedLoop._demod = self

    def setSymbolListener(self, listener):
        self.mSymbolListener = listener

    def receive(self, samples):
        """PSKDemodulator.receive(ReusableComplexBuffer): broadcasts one Dibit per decoded symbol"""
        samples = native.f32(samples)
        n = samples.size // 2
        if self._bank is None:
            self._length = n
            self._bank = Bank(1, self.mPLL.mSampleRate, self.KIND, block_size=n, max_samples_per_call=n,
                              symbol_rate=self.mPLL.mSymbolRate, pll_bandwidth=self.mPLL.mPLLBandwidth.value,
                              sample_counter_gain=self.mBuffer.mSampleCounterGain)
        elif n != self._length:
            raise native.IllegalArgumentException("buffer length changed; GPU-backed demodulators need fixed-size buffers")
        dibits = self._bank.process(samples.reshape(1, -1))[0]
        if self.mSymbolListener is not None:
            for d in dibits:
                self.mSymbolListener(Dibit(int(d)))
        return dibits


class DQPSKDecisionDirectedDemodulator(_PSKDemodulator):
    KIND = native.DEMOD_DQPSK_DECISION


class DQPSKGardnerDemodulator(_PSKDemodulator):
    KIND = native.DEMOD_DQPSK_GARDNER
