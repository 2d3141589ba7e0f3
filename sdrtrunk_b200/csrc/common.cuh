// Shared plumbing for libsdrgpu: status/error reporting, CUDA call checking, launch accounting.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <string>

#include "../../include/sdrgpu.h"

namespace sdrgpu {

extern thread_local std::string g_last_error;
extern std::atomic<uint64_t> g_launches;
extern int g_tuning[SDRGPU_TUNE_COUNT];   // sdrgpu_set_tuning

// dynamic shared memory a launch has to ask for so that at most `ctas` CTAs of it fit on one SM (228 KB per SM, 1 KB
// reserved per CTA); never less than `need`.  0 CTAs = no limit.
inline size_t smem_for_ctas_per_sm(size_t need, size_t static_bytes, int ctas)
{
    if (ctas <= 0) return need;
    const size_t per = (228 * 1024) / (size_t)(ctas + 1) + 1024;   // one more CTA of this size no longer fits
    const size_t want = per > static_bytes + 1024 ? per - static_bytes - 1024 : 0;
    const size_t cap = 227 * 1024 - static_bytes;
    const size_t v = want > need ? want : need;
    return v > cap ? cap : v;
}

inline sdrgpu_status fail(sdrgpu_status code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define SDRGPU_CUDA(call)                                                                         \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return ::sdrgpu::fail(SDRGPU_ERR_CUDA, "%s failed: %s (%s:%d)", #call,                \
                                  cudaGetErrorString(e__), __FILE__, __LINE__);                   \
    } while (0)

#define SDRGPU_TRY(expr)                      \
    do {                                      \
        sdrgpu_status s__ = (expr);           \
        if (s__ != SDRGPU_OK) return s__;     \
    } while (0)

// number of output rows the channelizer currently selects (channelizer.cu)
int chan_selected_count(const sdrgpu_channelizer *h);
// channelizer internals the fused pipeline (bank.cu) drives directly.  chan_enqueue writes channel-layout row c to
// d_out + c * stride, or, given a row table (a pipeline routing the rows to several banks), to rows[c] + col (floats)
sdrgpu_status chan_enqueue(sdrgpu_channelizer *h, const float2 *d_in, int n_in, float *d_out, long long stride, int layout,
                           int *n_blocks_out, float *const *rows = nullptr, long long col = 0);
cudaStream_t chan_stream(const sdrgpu_channelizer *h);
// host-buffer staging of the chunked paths: enqueue the H2D copy of complex samples [first, first + n) of the caller's
// buffer (in the handle's input format) on copy_stream; then, on the handle's stream, convert them to float I/Q if the
// format is a native one.  chan_convert returns the device float2 pointer of the chunk.
sdrgpu_status chan_upload(sdrgpu_channelizer *h, const void *iq, size_t first, int n, cudaStream_t copy_stream);
const float2 *chan_convert(sdrgpu_channelizer *h, const void *iq_device_or_null, size_t first, int n);
size_t chan_complex_bytes(const sdrgpu_channelizer *h);   // bytes of one complex sample in the handle's input format
int chan_half(const sdrgpu_channelizer *h);
void chan_swap_staging(sdrgpu_channelizer *h);   // host-input staging buffers alternate between the calls of an asynchronous pipeline
const void *chan_staging(const sdrgpu_channelizer *h);
cudaStream_t chan_osc_stream(const sdrgpu_channelizer *h);   // nullptr without frequency-corrected channels (call traces)
sdrgpu_status chan_osc_ahead(sdrgpu_channelizer *h);   // frequency-corrected channels: produce the next call's oscillator values now
void chan_set_throttled(sdrgpu_channelizer *h, bool on);   // next launches share the GPU with the demodulator (SDRGPU_TUNE_PFB_CTAS_PER_SM)
int chan_max_in(const sdrgpu_channelizer *h);
int chan_leftover(const sdrgpu_channelizer *h);  // samples buffered that did not fill a block yet (mSampleBufferPointer)   // complex samples one process call may carry (max_input_floats / 2)

// Airspy raw-sample converter (airspy.cu), stand-alone (sdrgpu_airspy_*) and as a channelizer input format
sdrgpu_status airspy_create(sdrgpu_airspy **out, int max_samples);
void airspy_destroy(sdrgpu_airspy *a);
size_t airspy_raw_bytes(int n_samples, int packed);
sdrgpu_status airspy_enqueue(sdrgpu_airspy *a, const uint8_t *d_raw, int n_samples, int packed, float2 *d_out, cudaStream_t stream);
sdrgpu_status airspy_reset(sdrgpu_airspy *a, cudaStream_t stream);

inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

// Optional per-handle kernel timing with CUDA events on the handle's stream.
struct KernelTimer {
    cudaEvent_t start = nullptr, stop = nullptr;
    bool enabled = false, pending = false;
    sdrgpu_status enable(bool on)
    {
        if (on && !start) {
            SDRGPU_CUDA(cudaEventCreate(&start));
            SDRGPU_CUDA(cudaEventCreate(&stop));
        }
        enabled = on;
        return SDRGPU_OK;
    }
    void begin(cudaStream_t s)
    {
        if (enabled) cudaEventRecord(start, s);
    }
    void end(cudaStream_t s)
    {
        if (enabled) {
            cudaEventRecord(stop, s);
            pending = true;
        }
    }
    sdrgpu_status read(float *ms)
    {
        *ms = 0.0f;
        if (!enabled || !pending) return SDRGPU_OK;
        SDRGPU_CUDA(cudaEventSynchronize(stop));
        SDRGPU_CUDA(cudaEventElapsedTime(ms, start, stop));
        return SDRGPU_OK;
    }
    ~KernelTimer()
    {
        if (start) cudaEventDestroy(start);
        if (stop) cudaEventDestroy(stop);
    }
};

}  // namespace sdrgpu
