/*
 * sdrgpu.h -- C ABI of libsdrgpu.so: the B200 (sm_100a) implementation of sdrtrunk's data-parallel DSP
 * hot path.  These entry points are what sdrtrunk's Java classes bind through java.lang.foreign
 * (INTEGRATION.md shows the binding); each group cites the reference class it replaces
 * ("J/" = src/main/java/io/github/dsheirer/ in smyers119/sdrtrunk).
 *
 * Conventions
 *  - every call returns an sdrgpu_status (0 = OK); sdrgpu_last_error() gives the message for the calling
 *    thread.  Nothing throws or aborts across the boundary.
 *  - all sample data is IEEE float32, complex data interleaved I,Q (the reference's float[] buffers).
 *  - `mem` arguments say where a caller pointer lives: SDRGPU_HOST (pageable or pinned host memory) or
 *    SDRGPU_DEVICE (device memory of the handle's GPU).  The library never keeps a caller pointer after
 *    the call returns (one exception, by name: sdrgpu_pipeline_submit_multi); host outputs are complete on return, device outputs are stream-ordered on the
 *    handle's stream (sdrgpu_*_sync or the caller's own stream sync).
 *  - a handle is bound to the device that was current in sdrgpu_init, owns its device state (filter
 *    history, PLL, timing) and is NOT thread safe: one host thread <-> one handle <-> one CUDA stream.
 *    Different handles are fully concurrent.
 *  - there is no CPU fallback: without a usable GPU every compute entry point returns SDRGPU_ERR_CUDA.
 */
#ifndef SDRGPU_H
#define SDRGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int sdrgpu_status;
enum {
    SDRGPU_OK = 0,
    SDRGPU_ERR_INVALID_ARG = 1, /* Java: IllegalArgumentException */
    SDRGPU_ERR_BAD_STATE = 2,   /* Java: IllegalStateException */
    SDRGPU_ERR_CUDA = 3,        /* CUDA runtime / no device */
    SDRGPU_ERR_OVERFLOW = 4,    /* more input than the handle was sized for (reference: queue OVERFLOW state) */
    SDRGPU_ERR_DESIGN = 5,      /* Java: FilterDesignException */
    SDRGPU_ERR_NOMEM = 6
};

enum { SDRGPU_HOST = 0, SDRGPU_DEVICE = 1 };

/* ------------------------------------------------------------------ runtime */
sdrgpu_status sdrgpu_init(int device);
const char *sdrgpu_last_error(void);
const char *sdrgpu_version(void);
sdrgpu_status sdrgpu_device_count(int *count);
sdrgpu_status sdrgpu_alloc_pinned(void **ptr, size_t bytes);
sdrgpu_status sdrgpu_free_pinned(void *ptr);
sdrgpu_status sdrgpu_device_alloc(void **ptr, size_t bytes);
sdrgpu_status sdrgpu_device_free(void *ptr);
sdrgpu_status sdrgpu_memcpy(void *dst, const void *src, size_t bytes, int dst_mem, int src_mem);
sdrgpu_status sdrgpu_device_synchronize(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t sdrgpu_launch_count(void);
/* Process-wide tuning knobs (launch shapes only: results never depend on them).  Unknown knob -> INVALID_ARG.
 *   FIR_CTAS_PER_SM / PFB_CTAS_PER_SM: resident CTAs per SM of fir_agc_kernel / pfb2_kernel while a pipeline runs its
 *   time chunks concurrently with the symbol demodulator (0 = whatever fits).  The demodulator is bound by the latency of
 *   its per-symbol feedback chain; every other resident warp on its scheduler delays each of its dependent instructions,
 *   so the filter kernels that overlap it are held to a few warps per scheduler.
 *   FIR_TILES_PER_CTA: consecutive assembler buffers of a channel one CTA of the FIR kernels filters (0 = chosen from the
 *   bank size: up to 4 while the grid still fills the GPU a dozen times over). */
enum { SDRGPU_TUNE_FIR_CTAS_PER_SM = 0, SDRGPU_TUNE_PFB_CTAS_PER_SM = 1, SDRGPU_TUNE_THROTTLE_ALWAYS = 2,
       SDRGPU_TUNE_FIR_TILES_PER_CTA = 3, SDRGPU_TUNE_COUNT = 8 };
sdrgpu_status sdrgpu_set_tuning(int knob, int value);
int sdrgpu_get_tuning(int knob);

/* ------------------------------------------------------------------ filter design (host side, runs once)
 * J/dsp/filter/FilterFactory.java:755-770 (getSincM2Synthesizer), :808-920 (getSincM2Channelizer),
 * :1007-1036 (getHalfBand); J/dsp/filter/Window.java.  `out` receives the taps, return value through
 * *n_taps.  The Java shim may instead pass taps designed by the unchanged FilterFactory. */
enum { SDRGPU_WINDOW_HAMMING = 0, SDRGPU_WINDOW_BLACKMAN = 1 };
sdrgpu_status sdrgpu_design_sinc_m2_channelizer(double channel_bandwidth, int channels, int taps_per_channel,
                                                float *out, int capacity, int *n_taps);
sdrgpu_status sdrgpu_design_sinc_m2_synthesizer(double channel_sample_rate, double channel_bandwidth, int channels,
                                                int taps_per_channel, float *out, int capacity, int *n_taps);
sdrgpu_status sdrgpu_design_half_band(int length, int window, float *out);
/* The decoders' baseband low-pass filters: FIRFilterSpecification.lowPassBuilder()...build() + FilterFactory.getTaps
 * (J/dsp/filter/fir/FIRFilterSpecification.java:381-428, J/dsp/filter/fir/remez/RemezFIRFilterDesigner.java:52-672,
 * J/dsp/filter/FilterFactory.java:671-681).  Frequencies in Hz, ripples in dB as the builder takes them; order < 6 =
 * estimate it (estimateFilterOrder, :909-937); odd_length: -1 = not requested, 0 / 1 = oddLength(false / true).
 * P25P1DecoderC4FM.java:136-148 = (50000, 5100, 6500, 0.01, 0.01, 0, -1, 16) -> 72 taps; P25P2DecoderHDQPSK.java:155-166 =
 * (50000, 6500, 7200, 0.005, 0.01, 0, -1, 16) -> 154 taps; NBFMDecoder.java:306-325 = (2 * 25000, 10000, 12500, 0.01,
 * 0.005, 0, 1, 16) -> 45 taps.  SDRGPU_ERR_DESIGN where getTaps returns null (no convergence). */
int sdrgpu_design_remez_estimate_order(double sample_rate, double frequency1, double frequency2, double pass_ripple_db,
                                       double stop_ripple_db);
sdrgpu_status sdrgpu_design_remez_low_pass(double sample_rate, double pass_band_end, double stop_band_start,
                                           double pass_ripple_db, double stop_ripple_db, int order, int odd_length,
                                           int grid_density, float *out, int capacity, int *n_taps);
/* ComplexPolyphaseChannelizerM2.getChannelCount (J/dsp/filter/channelizer/ComplexPolyphaseChannelizerM2.java:148-161) */
int sdrgpu_channel_count_for_rate(double sample_rate);

/* ------------------------------------------------------------------ channel calculator (host side)
 * J/dsp/filter/channelizer/ChannelCalculator.java:223-281 (getChannelIndexes), :515-541
 * (getCenterFrequencyForIndexes).  SDRGPU_ERR_INVALID_ARG where the Java throws IllegalArgumentException. */
sdrgpu_status sdrgpu_channel_indexes(double sample_rate, int channel_count, double center_frequency,
                                     long long channel_frequency, int channel_bandwidth, int *indexes,
                                     int capacity, int *n_indexes);
sdrgpu_status sdrgpu_center_frequency_for_indexes(double sample_rate, int channel_count, double center_frequency,
                                                  const int *indexes, int n_indexes, long long *frequency);

/* ------------------------------------------------------------------ tuner sample formats
 * The native formats the tuner converters turn into float I/Q before the channelizer: unsigned 8-bit
 * (J/source/tuner/usb/converter/ByteSampleConverter.java:21-35: (x - 127) / 128.0f), signed 8-bit
 * (SignedByteSampleConverter.java:21-35: x / 128.0f), little-endian signed 16-bit
 * (J/sample/ConversionUtils.java:22-34: x / 32767.0f).  Converting on the device cuts the host-to-device copy to
 * 1-2 bytes per value instead of 4. */
enum {
    SDRGPU_FORMAT_F32 = 0,
    SDRGPU_FORMAT_U8 = 1,
    SDRGPU_FORMAT_S8 = 2,
    SDRGPU_FORMAT_S16LE = 3,
    /* Airspy native buffers: 12-bit REAL samples at twice the complex rate, two bytes per sample little-endian or
     * "sample packing" (two samples in three bytes).  Stateful (DC removal + Hilbert transform, see sdrgpu_airspy
     * below): accepted by sdrgpu_chan_set_input_format only; n_floats of a process call then counts real samples,
     * which is also the number of floats of the I/Q stream they become. */
    SDRGPU_FORMAT_AIRSPY_U16LE = 4,
    SDRGPU_FORMAT_AIRSPY_PACKED12 = 5
};
/* n_values sample values (I and Q count separately) from src (format U8 / S8 / S16LE) to float dst */
sdrgpu_status sdrgpu_convert_samples(int format, const void *src, int src_mem, int n_values, float *dst, int dst_mem);

/* AirspySampleConverter (J/source/tuner/airspy/AirspySampleConverter.java:27-158): unpack -> DCRemovalFilter(0.01f)
 * (J/dsp/filter/dc/DCRemovalFilter.java:52-67) -> HilbertTransform.filter (J/dsp/filter/hilbert/HilbertTransform.java:
 * 88-132, coefficients from Filters.HALF_BAND_FILTER_47T).  Bit-exact with the Java: the sequential DC recursion is
 * run speculatively in 2 048-sample segments and verified (airspy.cu).  State (DC average, the Hilbert filter's last 47
 * samples, the fs/2 sign) carries over from call to call as in the Java object. */
typedef struct sdrgpu_airspy sdrgpu_airspy;
sdrgpu_status sdrgpu_airspy_create(sdrgpu_airspy **a, int max_samples);   /* real samples per call, even */
sdrgpu_status sdrgpu_airspy_destroy(sdrgpu_airspy *a);
sdrgpu_status sdrgpu_airspy_set_sample_packing(sdrgpu_airspy *a, int enabled);   /* AirspySampleConverter.setSamplePacking */
/* n_samples (even) raw samples -> n_samples floats of interleaved I/Q (n_samples / 2 complex samples) */
sdrgpu_status sdrgpu_airspy_convert(sdrgpu_airspy *a, const void *raw, int raw_mem, int n_samples, float *iq, int iq_mem);
/* diagnostics since creation: segments redone in parallel because their speculative start had not merged yet
 * (slowly varying input), and segments still inconsistent after that, which made a call fall back to one sequential
 * thread (noiseless constant / periodic input; expected 0 with ADC noise present) */
sdrgpu_status sdrgpu_airspy_repaired(sdrgpu_airspy *a, int *count);
sdrgpu_status sdrgpu_airspy_mismatches(sdrgpu_airspy *a, int *count);

/* ------------------------------------------------------------------ polyphase channelizer
 * Replaces ComplexPolyphaseChannelizerM2.receive + process + IFFTProcessor
 * (J/dsp/filter/channelizer/ComplexPolyphaseChannelizerM2.java:190-235,337-383,407-428) and, in channel
 * layout, the per-channel extraction of ReusableChannelResultsBuffer.getChannel +
 * One/TwoChannelOutputProcessor.process (J/sample/buffer/ReusableChannelResultsBuffer.java:112-153,
 * J/dsp/filter/channelizer/output/OneChannelOutputProcessor.java:81-106,
 * TwoChannelOutputProcessor.java:98-121). */
typedef struct sdrgpu_channelizer sdrgpu_channelizer;

/* taps: prototype low-pass, n_taps = channel_count * taps_per_channel (as ComplexPolyphaseChannelizerM2(float[]
 * taps, int sampleRate, int channelCount), :93-106); channel_count must be even.  max_input_floats sizes the
 * device staging for one process call (SDRGPU_ERR_OVERFLOW beyond it). */
sdrgpu_status sdrgpu_chan_create(sdrgpu_channelizer **h, const float *taps, int n_taps, int channel_count,
                                 int max_input_floats);
sdrgpu_status sdrgpu_chan_destroy(sdrgpu_channelizer *h);
/* run this handle's work on a caller-owned cudaStream_t (NULL = the handle's own stream) */
sdrgpu_status sdrgpu_chan_set_stream(sdrgpu_channelizer *h, void *cuda_stream);
sdrgpu_status sdrgpu_chan_sync(sdrgpu_channelizer *h);

/* tuner sample rate in Hz (the sampleRate argument of the ComplexPolyphaseChannelizerM2 constructors / setRates,
 * :93,114,169): needed before two-bin or frequency-corrected channels are selected (channel rate = 2 * rate / M) */
sdrgpu_status sdrgpu_chan_set_sample_rate(sdrgpu_channelizer *h, double sample_rate);

/* format of the `iq` buffers of sdrgpu_chan_process / sdrgpu_pipeline_process (default SDRGPU_FORMAT_F32): with a
 * native format `iq` points at the raw bytes and n_floats still counts sample values */
sdrgpu_status sdrgpu_chan_set_input_format(sdrgpu_channelizer *h, int format);

/* One output channel of the channel layout: one polyphase bin (bin2 < 0; OneChannelOutputProcessor) or two
 * adjacent bins recombined (TwoChannelOutputProcessor); frequency_offset_hz drives the frequency-correction
 * oscillator (ChannelOutputProcessor.setFrequencyOffset, :91-95); gain as PolyphaseChannelManager passes it
 * (= channel count, J/dsp/filter/channelizer/PolyphaseChannelManager.java:198-222). */
typedef struct {
    int bin1;
    int bin2;
    long long frequency_offset_hz;
    double gain;
} sdrgpu_output_channel;

/* select the output channels (default after create: every bin 0..M-1 as a one-bin channel with gain M and no
 * offset).  synthesis_filter (may be NULL if no two-bin channel) = getSincM2Synthesizer taps.  Two-bin channels run
 * TwoChannelSynthesizerM2 + FS4DownConverter + the frequency-correction Oscillator (always, as
 * TwoChannelOutputProcessor.java:113 does); one-bin channels run the Oscillator only with a non-zero offset
 * (OneChannelOutputProcessor.java:92-95).  Selecting resets the oscillators and synthesizer histories. */
sdrgpu_status sdrgpu_chan_select(sdrgpu_channelizer *h, const sdrgpu_output_channel *channels, int n_channels,
                                 const float *synthesis_filter, int n_synthesis_taps);

enum {
    SDRGPU_LAYOUT_RESULTS = 0, /* [n_blocks][2*M] floats: ReusableChannelResultsBuffer, all bins, no gain */
    SDRGPU_LAYOUT_CHANNELS = 1 /* [n_selected][out_stride_floats]: contiguous per-channel streams, gain applied */
};
/* Feeds n_floats interleaved I/Q floats of tuner samples (any length; block framing carries over between
 * calls like mSampleBufferPointer, :202-227).  *n_blocks receives the number of output blocks
 * (= complex samples per output channel) produced by this call.  out_stride_floats is only used by the
 * channel layout (row pitch in floats, >= 2 * blocks). */
sdrgpu_status sdrgpu_chan_process(sdrgpu_channelizer *h, const void *iq, int n_floats, int in_mem, float *out,
                                  long long out_stride_floats, int out_mem, int layout, int *n_blocks);
/* how many blocks a call with n_floats would produce now */
int sdrgpu_chan_blocks_for(const sdrgpu_channelizer *h, int n_floats);
/* device time of the dominant kernel of the last process call, measured with CUDA events on the handle's
 * stream (ms); enable first with sdrgpu_chan_enable_timing(h, 1) */
sdrgpu_status sdrgpu_chan_enable_timing(sdrgpu_channelizer *h, int enable);
sdrgpu_status sdrgpu_chan_last_kernel_ms(sdrgpu_channelizer *h, float *ms);

/* ------------------------------------------------------------------ per-channel banks
 * A bank runs the same per-channel chain over n_channels independent channel streams:
 *   [half-band decimation cascade] -> [complex FIR] -> [block AGC] -> demodulator
 * replacing, per channel, IComplexDecimationFilter (J/dsp/filter/decimate/DecimationFilterFactory.java:36-104,
 * J/dsp/filter/halfband/complex/ComplexHalfBandDecimationFilter.java:66-123), ComplexFIRFilter2.filter
 * (J/dsp/filter/fir/complex/ComplexFIRFilter2.java:112-129), ComplexFeedForwardGainControl.filter
 * (J/dsp/gain/ComplexFeedForwardGainControl.java:147-181), and one of FMDemodulator / SquelchingFMDemodulator
 * (J/dsp/fm/FMDemodulator.java:62-96, SquelchingFMDemodulator.java:63-101), DQPSKDecisionDirectedDemodulator
 * (J/dsp/psk/DQPSKDecisionDirectedDemodulator.java:50-89) or DQPSKGardnerDemodulator
 * (J/dsp/psk/DQPSKGardnerDemodulator.java:48-89) with CostasLoop + InterpolatingSampleBuffer. */
typedef struct sdrgpu_bank sdrgpu_bank;

enum {
    SDRGPU_DEMOD_NONE = 0,              /* filters only: output = filtered (gain-controlled) complex stream */
    SDRGPU_DEMOD_FM = 1,                /* FMDemodulator */
    SDRGPU_DEMOD_FM_SQUELCH = 2,        /* SquelchingFMDemodulator */
    SDRGPU_DEMOD_DQPSK_DECISION = 3,    /* DQPSKDecisionDirectedDemodulator (C4FM, DMR) */
    SDRGPU_DEMOD_DQPSK_GARDNER = 4      /* DQPSKGardnerDemodulator (LSM, Phase 2 HDQPSK) */
};

typedef struct {
    int n_channels;
    double sample_rate;        /* of the incoming channel streams (Hz) */
    int decimation;            /* 0 (none), 2, 4, ... 1024 */
    const float *fir_taps;     /* NULL / 0 = no FIR (P25P1DecoderLSM.filter returns its input) */
    int n_fir_taps;
    float fir_gain;            /* ComplexFIRFilter2 gain, 1.0f default */
    int agc;                   /* 1 = ComplexFeedForwardGainControl per block_size-sample buffer */
    int block_size;            /* assembler buffer in complex samples; 1024 (PolyphaseChannelSource.java:42) */
    int demod;                 /* SDRGPU_DEMOD_* */
    double symbol_rate;        /* DQPSK: 4800 / 6000 */
    double pll_bandwidth;      /* DQPSK: PLLBandwidth loop bandwidth 400/300/250/200 */
    float sample_counter_gain; /* DQPSK: 0.3 (P1) / 0.1 (P2) */
    float fm_gain;             /* FM: FMDemodulator gain */
    double squelch_alpha;      /* FM_SQUELCH: 0.0004 */
    double squelch_threshold_db; /* FM_SQUELCH: -78.0 */
    int squelch_ramp;          /* FM_SQUELCH: 4 */
    int max_samples_per_call;  /* per channel, complex samples; sizes device staging */
} sdrgpu_bank_config;

/* presets of the reference's decoder front-ends (chain order + constants):
 * P25P1DecoderC4FM.java:62-93, P25P1DecoderLSM.java:67-106, P25P2DecoderHDQPSK.java:62-110,
 * NBFMDecoder.java:55-62,262-349 */
enum {
    SDRGPU_PRESET_P25_C4FM = 0,
    SDRGPU_PRESET_P25_LSM = 1,
    SDRGPU_PRESET_P25_HDQPSK = 2,
    SDRGPU_PRESET_NBFM = 3,
    SDRGPU_PRESET_DMR = 4 /* J/module/decode/dmr/DMRDecoder.java:58-131: FIR -> AGC -> decision-directed, BW_300, gain 0.4 */
};
sdrgpu_status sdrgpu_bank_config_preset(sdrgpu_bank_config *cfg, int preset, int n_channels, double sample_rate,
                                        const float *fir_taps, int n_fir_taps, int max_samples_per_call);

sdrgpu_status sdrgpu_bank_create(sdrgpu_bank **b, const sdrgpu_bank_config *cfg);
sdrgpu_status sdrgpu_bank_destroy(sdrgpu_bank *b);
sdrgpu_status sdrgpu_bank_set_stream(sdrgpu_bank *b, void *cuda_stream);
sdrgpu_status sdrgpu_bank_sync(sdrgpu_bank *b);

/* Feeds n_samples complex samples per channel: channel c starts at iq + c * in_stride_floats.
 * Outputs (each may be NULL; `out_mem` applies to all of them):
 *   symbols  [n_channels][symbol_stride] one byte per decoded Dibit (Dibit.getValue 0..3, J/dsp/symbol/Dibit.java:27-30);
 *            FM_SQUELCH banks with squelch reporting on: one status byte per assembler buffer (see
 *            sdrgpu_bank_set_squelch_reporting); other banks ignore it
 *   demod    [n_channels][demod_stride_floats] float: FM demodulated samples (FM demods) or the filtered /
 *            gain-controlled interleaved complex stream (SDRGPU_DEMOD_NONE, and as a tap point for DQPSK)
 *   counts   [n_channels] number of symbols (DQPSK) or floats (otherwise) written per channel by this call
 * With agc / DQPSK the chain consumes whole block_size buffers only (the assembler framing,
 * ReusableComplexBufferAssembler.java:99-167); a remainder stays buffered in the handle. */
sdrgpu_status sdrgpu_bank_process(sdrgpu_bank *b, const float *iq, long long in_stride_floats, int n_samples,
                                  int in_mem, uint8_t *symbols, int symbol_stride, float *demod,
                                  long long demod_stride_floats, int *counts, int out_mem);
/* IPhaseLockedLoop.correctInversion / reset (J/dsp/psk/pll/CostasLoop.java:91-104,224-229): applied at the next
 * buffer boundary of that channel (host-driven sync feedback, SURVEY.md hard part 4) */
sdrgpu_status sdrgpu_bank_correct_inversion(sdrgpu_bank *b, int channel, double radians);
sdrgpu_status sdrgpu_bank_reset_pll(sdrgpu_bank *b, int channel);
/* Sync-pattern detection and the PLL phase-inversion feedback it drives, on the device, per channel:
 * P25P1SyncDetector (J/module/decode/p25/phase1/P25P1SyncDetector.java:37-168: MultiSyncPatternMatcher over 48 bits,
 * SoftSyncDetector(P25_PHASE1_NORMAL, 4 bit errors), exact detectors for the 90 CW / 90 CCW / 180 degree rotated
 * patterns that call IPhaseLockedLoop.correctInversion(+-2 pi 1200 / fs, 2 pi 2400 / fs)) behind the 33-dibit delay
 * buffer of P25P1DataUnitDetector.java:41,106; or P25P2SyncDetector (40 bits, J/module/decode/p25/phase2/
 * P25P2SyncDetector.java:40-160) behind the 160-dibit delay of P25P2SuperFrameDetector.java:66,159.  The correction
 * is applied at exactly the symbol the reference applies it (after that symbol's CostasLoop.adjust), not at the next
 * buffer boundary.  The detector is fed every dibit, as the reference's framers feed it while they search for sync
 * (they pause it while a message is being assembled / fragment sync is held; that framing stays on the host).
 * With a detector enabled every symbol byte is  dibit | event << 2 | bit_errors << 5 :
 * the event the detector raised at that symbol (syncDetected / correctInversion / syncLost) and, for
 * SDRGPU_SYNC_EVENT_SYNC, the number of bit errors passed to ISyncDetectListener.syncDetected.
 * Enabling (or re-enabling) starts from a fresh detector on every channel. */
enum { SDRGPU_SYNC_NONE = 0, SDRGPU_SYNC_P25_PHASE1 = 1, SDRGPU_SYNC_P25_PHASE2 = 2, SDRGPU_SYNC_P25_PHASE2_FRAMED = 3 };
/* SDRGPU_SYNC_P25_PHASE2_FRAMED runs the reference's complete Phase 2 framing per channel instead of the bare
 * detector: P25P2SuperFrameDetector (J/module/decode/p25/phase2/P25P2SuperFrameDetector.java:132-302), i.e. the
 * fragment-sync state machine (sync patterns at dibits 360 and 540 of the 720-dibit fragment, 10 / 4 bit errors),
 * its sync-loss accounting, and the P25P2SyncDetector with the PLL inversion detectors, fed -- as in the Java -- only
 * while fragment sync is lost.  P25P2MessageFramer.receive hands every dibit to that class, so nothing is gated from
 * outside and the result is exact.  Symbol bytes are then  dibit | events << 2  with the SDRGPU_P2_EVENT_* bits: the
 * host cuts a super-frame fragment (the last 720 dibits) wherever SDRGPU_P2_EVENT_FRAGMENT is set. */
enum {
    SDRGPU_P2_EVENT_FRAGMENT = 1,      /* broadcastFragment */
    SDRGPU_P2_EVENT_SYNC_LOSS = 2,     /* broadcastSyncLoss */
    SDRGPU_P2_EVENT_INVERSION = 4,     /* correctInversion applied; bits 3-4: 1 = 90 CW, 2 = 90 CCW, 3 = 180 */
    SDRGPU_P2_EVENT_SYNCHRONIZED = 32  /* mSynchronized after this dibit */
};
enum {
    SDRGPU_SYNC_EVENT_NONE = 0,
    SDRGPU_SYNC_EVENT_SYNC = 1,             /* primary pattern within 4 bit errors */
    SDRGPU_SYNC_EVENT_INVERSION_90_CW = 2,  /* rotated pattern matched exactly: loop frequency corrected */
    SDRGPU_SYNC_EVENT_INVERSION_90_CCW = 3,
    SDRGPU_SYNC_EVENT_INVERSION_180 = 4,
    SDRGPU_SYNC_EVENT_LOST = 5              /* MultiSyncPatternMatcher: more than the loss threshold of bits without a match */
};
sdrgpu_status sdrgpu_bank_set_sync_detector(sdrgpu_bank *b, int kind);
/* Tuning: how many lanes of a warp work on one channel in the symbol demodulator kernel -- 32 (one warp per channel),
 * 16 (two channels per warp), 8 / 4 / 2 (four / eight / sixteen channels per warp, several samples of a symbol period per
 * lane; with a sync detector: 8 / 4 for Phase 1 sync and for Phase 2 sync behind the Gardner demodulator, other
 * combinations run two channels per warp), 1 (one thread per channel), 0 = chosen from the bank size (default).  All variants do
 * the same arithmetic on the same per-channel state; the result does not depend on the choice, which may change
 * between calls -- except while a sync detector (SDRGPU_SYNC_P25_PHASE1 / _PHASE2) is enabled: choose the layout first
 * (SDRGPU_ERR_BAD_STATE otherwise). */
sdrgpu_status sdrgpu_bank_set_demodulator_lanes(sdrgpu_bank *b, int lanes_per_channel);
/* Per-symbol tap points of ONE channel of the bank, the listeners of DQPSKDecisionDirectedDemodulatorInstrumented /
 * DQPSKGardnerDemodulatorInstrumented (J/dsp/psk/DQPSKDecisionDirectedDemodulatorInstrumented.java:74-108: complex symbol,
 * samples per symbol, PLL error, PLL frequency).  While a tap is set (channel >= 0; -1 clears it) every process call also
 * demodulates that channel from a copy of its states on a side stream, recording per symbol 6 doubles
 * {symbol_i, symbol_q, detected samples per symbol, loop frequency in radians per sample, sampling point, PLL error} as
 * they are at the end of calculateSymbol(); the bank's own launch and results are not affected.
 * sdrgpu_bank_read_symbol_tap returns the symbols of the last process call (values[6 * capacity_symbols]). */
sdrgpu_status sdrgpu_bank_set_symbol_tap(sdrgpu_bank *b, int channel);
sdrgpu_status sdrgpu_bank_read_symbol_tap(sdrgpu_bank *b, double *values, int capacity_symbols, int *n_symbols);
/* Squelch state per assembler buffer, for SDRGPU_DEMOD_FM_SQUELCH banks: what NBFMDecoder asks its
 * SquelchingFMDemodulator after each demodulate(buffer) (isSquelchChanged, J/dsp/fm/SquelchingFMDemodulator.java;
 * PowerSquelch.java:88-159).  While reporting is on (default off), every process call -- sdrgpu_bank_process,
 * sdrgpu_pipeline_process / _multi, and sdrgpu_pipeline_process_routed through sdrgpu_bank_output.symbols -- writes one
 * status byte per assembler buffer it consumes into `symbols`: byte i of channel c at symbols[c * symbol_stride + i],
 * for i < counts[c] / (block_size / decimation) (a bank consumes whole buffers, so every call starts on a buffer
 * boundary).  Bits 0-1: the squelch state after the buffer's last sample (SDRGPU_SQUELCH_ATTACK .. _UNMUTE); bit 2,
 * SDRGPU_SQUELCH_CHANGED: the state changed at least once during the buffer (PowerSquelch.mSquelchChanged).  The
 * demodulated samples are 0.0f in MUTE and ATTACK.  symbols == NULL writes no statuses; a symbol_stride smaller than
 * the call's buffers gets INVALID_ARG before any device work.  With reporting off `symbols` is not touched.  Any other
 * bank gets INVALID_ARG, with nothing changed. */
enum {
    SDRGPU_SQUELCH_ATTACK = 0,
    SDRGPU_SQUELCH_DECAY = 1,
    SDRGPU_SQUELCH_MUTE = 2,
    SDRGPU_SQUELCH_UNMUTE = 3,
    SDRGPU_SQUELCH_CHANGED = 4
};
sdrgpu_status sdrgpu_bank_set_squelch_reporting(sdrgpu_bank *b, int enabled);
/* PowerSquelch.setSquelchThreshold per channel (channel = -1: every channel), in dB as squelch_threshold_db (the
 * configured value is every channel's initial one).  Used from the next buffer the bank processes; the squelch's IIR
 * and ramp state carry on.  INVALID_ARG for a bank without squelch, a channel out of range or a non-finite value. */
sdrgpu_status sdrgpu_bank_set_squelch_threshold(sdrgpu_bank *b, int channel, double threshold_db);
/* loop state tap points of one channel: {pll phase, pll frequency, sampling point, detected samples/symbol} */
sdrgpu_status sdrgpu_bank_get_loop_state(sdrgpu_bank *b, int channel, double *state4);
/* 4 dibits per byte MSB first (J/dsp/symbol/DibitToByteBufferAssembler.java:58-93); host helper */
int sdrgpu_pack_dibits(const uint8_t *dibits, int n, uint8_t *out);
sdrgpu_status sdrgpu_bank_enable_timing(sdrgpu_bank *b, int enable);
/* ms[0] = filter (decimate/FIR/AGC) kernels, ms[1] = demodulator kernel of the last process call */
sdrgpu_status sdrgpu_bank_last_kernel_ms(sdrgpu_bank *b, float *ms2);

/* ------------------------------------------------------------------ fused pipeline
 * channelizer -> bank without a host round trip: the channelizer's selected channels (in order) feed the
 * bank's channels; only symbols / demodulated floats come back.  Replaces the chain
 * PolyphaseChannelManager.BufferSourceEventMonitor.receive -> ... -> decoder.receive
 * (SURVEY.md section 3.2 / 3.3). */
typedef struct sdrgpu_pipeline sdrgpu_pipeline;
sdrgpu_status sdrgpu_pipeline_create(sdrgpu_pipeline **p, sdrgpu_channelizer *chan, sdrgpu_bank *bank);
sdrgpu_status sdrgpu_pipeline_destroy(sdrgpu_pipeline *p); /* does not destroy chan / bank; call it before theirs */
/* a process call is cut into `chunks` time chunks (default 8, behind a ramp of smaller leading chunks; 1 = single pass) so that copies, channelizer / filter
 * kernels and the latency-bound demodulator of successive chunks overlap; the results do not depend on it */
sdrgpu_status sdrgpu_pipeline_set_chunks(sdrgpu_pipeline *p, int chunks);
sdrgpu_status sdrgpu_pipeline_process(sdrgpu_pipeline *p, const void *iq, int n_floats, int in_mem,
                                      uint8_t *symbols, int symbol_stride, float *demod,
                                      long long demod_stride_floats, int *counts, int out_mem);

/* Several tuners, one bank.  In the reference every channel is its own task (TunerChannelSource.processSamples,
 * J/source/tuner/channel/TunerChannelSource.java:290-319, scheduled per channel by
 * PolyphaseChannelManager.java:582-623), whichever tuner it came from.  The symbol demodulator is serial per
 * channel, so one tuner's few hundred channels leave most of the GPU idle: a multi-tuner pipeline lets n_chans
 * channelizers (equal channel counts) write consecutive row ranges of ONE bank -- bank rows
 * [sum of the selections before k, ...) belong to chans[k] -- and the filter / demodulator kernels run once over all of
 * them.  iq[k] is tuner k's buffer (every tuner delivers n_floats values per call, in its channelizer's input
 * format); outputs are indexed by bank row.  Results are identical to n_chans single-tuner pipelines. */
sdrgpu_status sdrgpu_pipeline_create_multi(sdrgpu_pipeline **p, sdrgpu_channelizer *const *chans, int n_chans,
                                           sdrgpu_bank *bank);
sdrgpu_status sdrgpu_pipeline_process_multi(sdrgpu_pipeline *p, const void *const *iq, int n_floats, int in_mem,
                                            uint8_t *symbols, int symbol_stride, float *demod,
                                            long long demod_stride_floats, int *counts, int out_mem);
/* Asynchronous form for a continuous stream (host buffers in, dibits out; DQPSK banks).  A synchronous call cannot hide
 * its first H2D chunk nor the chain of its last one; a tuner delivers buffer after buffer (the reference's 5 ms cadence,
 * J/dsp/filter/channelizer/PolyphaseChannelManager.java:582-623), so the copies of buffer k + 1 can run while the kernels
 * of buffer k finish.  submit enqueues the call and returns; the caller must leave iq[...], symbols and counts alone until
 * the matching sdrgpu_pipeline_wait returns (the one documented exception to "the library never keeps a caller pointer").
 * At most two calls in flight (BAD_STATE beyond): submit(k + 1), then wait() -- which returns when the OLDEST call in
 * flight, k, has its outputs on the host -- with two alternating sets of host buffers.  Results are those of the same
 * sequence of sdrgpu_pipeline_process_multi calls.  wait with nothing in flight returns at once; process / process_multi
 * refuse to run while calls are in flight. */
sdrgpu_status sdrgpu_pipeline_submit_multi(sdrgpu_pipeline *p, const void *const *iq, int n_floats, uint8_t *symbols,
                                           int symbol_stride, int *counts);
sdrgpu_status sdrgpu_pipeline_wait(sdrgpu_pipeline *p);
/* time chunks for device-resident input, and for the asynchronous calls above (nothing to copy, but with many channels the
 * latency-bound demodulator of chunk i overlaps the FIR kernels of chunk i+1; the first chunks are a quarter and half a
 * chunk).  Default: by bank size -- 6 from 2400 channels (several tuners in one bank), else 1 */
sdrgpu_status sdrgpu_pipeline_set_device_chunks(sdrgpu_pipeline *p, int chunks);

/* Several tuners, several banks: one channelizer pass feeds banks of different decoder types (a tuner serving a P25
 * control channel, P25 traffic, DMR and NBFM channels at once, as PolyphaseChannelManager serves channels of every
 * decoder type from one channelizer).  route[r], one entry per selected channel in pipeline row order (chans[0]'s
 * selection in order, then chans[1]'s, ...), is the index in banks[] of the bank that decodes that channel; bank j's rows
 * are the rows routed to it, in that order.  Every bank must receive exactly its n_channels rows, all banks must have the
 * same block_size and no pending samples (they are kept in step), and the channelizers the same channel count
 * (INVALID_ARG / BAD_STATE, checked before any device work: a refused create leaves every handle usable).  While the
 * pipeline lives, every bank runs on banks[0]'s stream (sdrgpu_bank_set_stream; destroy restores the others').
 * sdrgpu_pipeline_create_multi is the one-bank, all-zero route of this.  outputs[j] takes bank j's outputs, as the
 * arguments of sdrgpu_pipeline_process_multi would; every bank runs the schedule it would run alone, and bank j's
 * results equal those of a one-bank pipeline whose channelizers select only bank j's channels.  A channelizer whose
 * selection no longer has the row count the route was built for gets BAD_STATE; so do sdrgpu_pipeline_process_multi and
 * sdrgpu_pipeline_submit_multi on a pipeline of several banks. */
typedef struct {
    uint8_t *symbols; int symbol_stride;          /* as sdrgpu_pipeline_process_multi, per bank */
    float *demod; long long demod_stride_floats;
    int *counts;
} sdrgpu_bank_output;
sdrgpu_status sdrgpu_pipeline_create_routed(sdrgpu_pipeline **p, sdrgpu_channelizer *const *chans, int n_chans,
                                            sdrgpu_bank *const *banks, int n_banks, const int *route);
sdrgpu_status sdrgpu_pipeline_process_routed(sdrgpu_pipeline *p, const void *const *iq, int n_floats, int in_mem,
                                             const sdrgpu_bank_output *outputs /* [n_banks] */, int out_mem);

#ifdef __cplusplus
}
#endif
#endif
