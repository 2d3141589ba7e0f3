// The channel filters of a bank (filters.cuh): the half-band decimation stages and the complex FIR + block AGC.
//
// Replaces, per channel (J/ = src/main/java/io/github/dsheirer/):
//   ComplexHalfBandDecimationFilter.decimateComplex   J/dsp/filter/halfband/complex/ComplexHalfBandDecimationFilter.java:66-123
//   ComplexFIRFilter2.filter / RealFIRFilter2.filter   J/dsp/filter/fir/complex/ComplexFIRFilter2.java:112-129, real/RealFIRFilter2.java:77-95
//   ComplexFeedForwardGainControl.filter               J/dsp/gain/ComplexFeedForwardGainControl.java:147-181
//
// Arithmetic contract: float ops are separately rounded (-fmad=false, __f*_rn) exactly where the Java has separate
// * and +; fmaf in tap order where the Java calls Math.fma.
#include <cstdint>

#include "filters.cuh"
#include "tma.cuh"

using namespace sdrgpu;

namespace {

// ---------------------------------------------------------------------------------------------------------------
// half-band decimate-by-2 stage.  in row: [L-1 history | n new], out row offset out_off, n/2 outputs.
//   out[m] = sum_{j even, j < (L-1)/2} c[j] * (x[2m + j] + x[2m + L-1-j])  (add, mul, add; ascending j)
//            + x[2m + (L-1)/2] * 0.5
// ---------------------------------------------------------------------------------------------------------------
__global__ void halfband_kernel(const float2 *__restrict__ in, long long in_stride, float2 *__restrict__ out,
                                long long out_stride, int out_off, int n_out, const __grid_constant__ HalfBandTaps taps)
{
    const int c = blockIdx.y;
    const float2 *x = in + (size_t)c * in_stride;
    float2 *y = out + (size_t)c * out_stride + out_off;
    const int L = taps.length, half = (L - 1) / 2;
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < n_out; m += gridDim.x * blockDim.x) {
        const float2 *p = x + 2 * m;
        float ai = 0.0f, aq = 0.0f;
        for (int j = 0; j < half; j += 2) {
            const float2 a = p[j], b = p[L - 1 - j];
            const float h = taps.c[j];
            ai = __fadd_rn(ai, __fmul_rn(h, __fadd_rn(a.x, b.x)));
            aq = __fadd_rn(aq, __fmul_rn(h, __fadd_rn(a.y, b.y)));
        }
        const float2 mid = p[half];
        ai = __fadd_rn(ai, __fmul_rn(mid.x, 0.5f));
        aq = __fadd_rn(aq, __fmul_rn(mid.y, 0.5f));
        y[m] = make_float2(ai, aq);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// FIR (+ block AGC).  One CTA per (channel, tile of <= 1024 samples); 128 threads x 8 consecutive outputs each.
//   y[n] = fma chain over k = 0..N-1 of x[n-k] * h[k], acc starting at 0.0f, then * gain          (RealFIRFilter2.java:77-95)
//   AGC: env = max(|i|,|q|) + 0.4f*min(|i|,|q|); g = 1.0f / max(1e-4f, max_n env); y *= g         (ComplexFeedForwardGainControl.java:147-181)
// The taps are padded with zeros to a multiple of 8 (kp); a thread keeps a 16-sample window of x in registers, runs
// 8 taps x 8 outputs x (I, Q) = 128 FFMA on it, then slides it by 8 samples with four LDS.128.  The window lives in
// shared memory at float2 index i + 2 * (i >> 3) (16 bytes of skew per 64): the 64-byte chunks of the 32 lanes then
// fall on distinct 16-byte bank groups.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kFirThreads = 128;
constexpr int kFirPer = 8;

__device__ __forceinline__ int skew8(int i) { return i + 2 * (i >> 3); }

// float2 slots of one skewed window of `window` samples, with 8 of slack, rounded up to whole 16-byte pairs
__host__ __device__ inline int fir_window_len(int window) { return (window + 2 * (window >> 3) + 8 + 1) & ~1; }

// ComplexFeedForwardGainControl's envelope of a sample: max(|i|, |q|) + 0.4f * min(|i|, |q|)
__device__ __forceinline__ float agc_envelope(float i, float q)
{
    const float a = fabsf(i), b = fabsf(q);
    return (a > b) ? __fadd_rn(a, __fmul_rn(0.4f, b)) : __fadd_rn(b, __fmul_rn(0.4f, a));
}

__device__ __forceinline__ void load8p(const float2 *group, float2 *w)   // group = xs + skew8(i), i a multiple of 8
{
    const float4 *p = reinterpret_cast<const float4 *>(group);
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const float4 v = p[q];
        w[2 * q] = make_float2(v.x, v.y);
        w[2 * q + 1] = make_float2(v.z, v.w);
    }
}

// 16-byte asynchronous global -> shared copies (LDGSTS): the window of the NEXT tile streams into the other half of a
// double buffer while this tile's taps run; no registers are staged and no warp waits on the fill
__device__ __forceinline__ void cp_async16(void *dst_shared, const void *src_global)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_shared)), "l"(src_global) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(kPending) : "memory"); }

// acc[j] = sum over taps of x[n0 + j - k] h[k], k ascending (the Java's tap order), kp a positive multiple of 8;
// wbase = skewed address of x[n0] (n0 a multiple of 8 within the window)
__device__ __forceinline__ void fir_taps8(const float2 *wbase, const float *hs, int kp, float2 (&acc)[kFirPer])
{
    // three rotating groups of 8 samples: a step of 8 taps needs x[n0 - k0 - 8 .. n0 - k0 + 7] = (lo, hi); the next
    // step's new group is loaded into the registers the current one no longer needs (no register moves).  A group of 8
    // samples is 10 skewed slots, so the window walks down by constant offsets from wbase (no index arithmetic per load)
    float2 ga[8], gb[8], gc[8];
    load8p(wbase, gc);
    load8p(wbase - 10, gb);
    // the I and Q rails of one output share a packed FFMA2 (sm_100 fma.rn.f32x2: two independent, correctly rounded
    // fused multiply-adds -- each rail is exactly Math.fma in tap order): half the FMA issue slots
#pragma unroll
    for (int j = 0; j < kFirPer; j++) acc[j] = make_float2(0.0f, 0.0f);
    // taps k0 .. k0 + 7 on (lo, hi): x[n0 + j - (k0 + u)] * h[k0 + u], u ascending
#define FIR_STEP(lo, hi, k0_)                                                                                   \
    {                                                                                                           \
        const float4 ha_ = *reinterpret_cast<const float4 *>(hs + (k0_));                                       \
        const float4 hb_ = *reinterpret_cast<const float4 *>(hs + (k0_) + 4);                                   \
        const float h_[8] = {ha_.x, ha_.y, ha_.z, ha_.w, hb_.x, hb_.y, hb_.z, hb_.w};                           \
        _Pragma("unroll") for (int u = 0; u < 8; u++) {                                                         \
            const float2 hh_ = make_float2(h_[u], h_[u]);                                                       \
            _Pragma("unroll") for (int j = 0; j < kFirPer; j++) {                                               \
                const float2 x_ = (j - u >= 0) ? hi[j - u] : lo[8 + j - u];                                     \
                acc[j] = __ffma2_rn(x_, hh_, acc[j]);                                                           \
            }                                                                                                   \
        }                                                                                                       \
    }
    // (loading an iteration's first taps during the previous iteration's last step -- the first FFMA2 of an iteration waits
    // for them, 2.6 % of the kernel's stall samples -- was measured: 96 registers with a spill, 0.7 % faster: not kept)
    int k0 = 0;
    for (; k0 + 24 <= kp; k0 += 24, wbase -= 30) {
        load8p(wbase - 20, ga);
        FIR_STEP(gb, gc, k0);
        load8p(wbase - 30, gc);
        FIR_STEP(ga, gb, k0 + 8);
        if (k0 + 24 < kp) load8p(wbase - 40, gb);
        FIR_STEP(gc, ga, k0 + 16);
    }
    if (k0 < kp) {   // 8 or 16 taps left
        if (k0 + 8 < kp) load8p(wbase - 20, ga);
        FIR_STEP(gb, gc, k0);
        if (k0 + 8 < kp) FIR_STEP(ga, gb, k0 + 8);
    }
#undef FIR_STEP
}

__global__ void __launch_bounds__(kFirThreads)
fir_agc_kernel(const float2 *__restrict__ in, long long in_stride, int in_off, float2 *__restrict__ out,
               long long out_stride, int tile, int n_total, int kp, float fir_gain, int agc, int tiles_per_cta,
               const __grid_constant__ FirTaps taps)
{
    extern __shared__ __align__(16) float2 xs_all[];   // two skewed windows: local i <-> stream sample blk*tile - kp + i
    __shared__ __align__(16) float hs[kMaxFirTaps];
    __shared__ float red[kFirThreads / 32];
    const int c = blockIdx.y, tid = threadIdx.x;
    const int window = kp + ((tile + 7) & ~7);
    const int wlen = fir_window_len(window);
    const int n_tiles = (n_total + tile - 1) / tile;
    const int first = blockIdx.x * tiles_per_cta, last = min(first + tiles_per_cta, n_tiles);
    const float2 *row = in + (size_t)c * in_stride + in_off;
    // rows, in_off, kp and (for more than one tile) tile are even: every pair of samples is a 16-byte aligned copy
    auto fill = [&](int blk, float2 *xs) {
        const float2 *src = row + (size_t)blk * tile - kp;
        const int valid = kp + min(tile, n_total - blk * tile);   // the last tile of a call may be partial (no AGC framing)
        if (valid == window) {
            // whole tile (the common case): a thread's copies are 256 samples apart, i.e. 320 skewed slots -- two pointer
            // increments per copy instead of the index arithmetic of the general loop below
            const float2 *s = src + 2 * tid;
            float2 *d = xs + skew8(2 * tid);
            for (int i = 2 * tid; i < window; i += 2 * kFirThreads, s += 2 * kFirThreads, d += 2 * kFirThreads + (kFirThreads >> 1))
                cp_async16(d, s);
        } else {
            for (int i = 2 * tid; i < window; i += 2 * kFirThreads) {
                float2 *dst = xs + skew8(i);
                if (i + 1 < valid) {
                    cp_async16(dst, src + i);
                } else {
                    dst[0] = i < valid ? src[i] : make_float2(0.f, 0.f);
                    dst[1] = make_float2(0.f, 0.f);
                }
            }
        }
        cp_async_commit();
    };
    for (int k = tid; k < kp; k += kFirThreads) hs[k] = taps.h[k];
    if (first < last) fill(first, xs_all);
    for (int blk = first; blk < last; blk++) {
    float2 *xs = xs_all + ((blk - first) & 1) * wlen;
    if (blk + 1 < last) {
        fill(blk + 1, xs_all + (((blk - first) & 1) ^ 1) * wlen);
        cp_async_wait<1>();
    } else {
        cp_async_wait<0>();
    }
    __syncthreads();
    const int block = min(tile, n_total - blk * tile);

    const int n0 = tid * kFirPer;   // first output of this thread (tile <= 1024 = 128 threads x 8)
    float ai[kFirPer], aq[kFirPer];
    if (n0 < block) {
        const float2 *wbase = xs + skew8(kp + n0);   // kp and n0 are multiples of 8
        if (kp > 0) {
            float2 acc[kFirPer];
            fir_taps8(wbase, hs, kp, acc);
#pragma unroll
            for (int j = 0; j < kFirPer; j++) {
                ai[j] = __fmul_rn(acc[j].x, fir_gain);
                aq[j] = __fmul_rn(acc[j].y, fir_gain);
            }
        } else {
            float2 x[kFirPer];
            load8p(wbase, x);
#pragma unroll
            for (int j = 0; j < kFirPer; j++) {
                ai[j] = x[j].x;
                aq[j] = x[j].y;
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < kFirPer; j++) {
            ai[j] = 0.0f;
            aq[j] = 0.0f;
        }
    }

    if (agc) {
        // one AGC buffer == one CTA (block <= 1024, asserted on the host)
        float m = 0.0001f;
#pragma unroll
        for (int j = 0; j < kFirPer; j++) {
            if (n0 + j < block) {
                const float env = agc_envelope(ai[j], aq[j]);
                if (env > m) m = env;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((tid & 31) == 0) red[tid >> 5] = m;
        __syncthreads();
        m = red[0];
#pragma unroll
        for (int wdx = 1; wdx < kFirThreads / 32; wdx++) m = fmaxf(m, red[wdx]);
        const float g = __fdiv_rn(1.0f, m);
#pragma unroll
        for (int j = 0; j < kFirPer; j++) {
            ai[j] = __fmul_rn(ai[j], g);
            aq[j] = __fmul_rn(aq[j], g);
        }
    }
    float2 *dst = out + (size_t)c * out_stride + (size_t)blk * tile + n0;
    if (n0 + kFirPer <= block && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
        for (int j = 0; j < kFirPer; j += 2) *reinterpret_cast<float4 *>(dst + j) = make_float4(ai[j], aq[j], ai[j + 1], aq[j + 1]);
    } else {
#pragma unroll
        for (int j = 0; j < kFirPer; j++)
            if (n0 + j < block) dst[j] = make_float2(ai[j], aq[j]);
    }
    __syncthreads();   // this window (and red[]) may be refilled two tiles from now
    }
}

// ---------------------------------------------------------------------------------------------------------------
// fir_agc_split_kernel: the same arithmetic as fir_agc_kernel for the decoders' common case (block AGC on, 1024-sample
// assembler buffers, whole buffers), without a block-wide barrier in the steady state.  fir_agc_kernel meets three
// __syncthreads per buffer (window landed / AGC maximum / buffers free), and a CTA's four warps sit on four different
// schedulers, each shared with five warps of other CTAs: 9 % of the warp time waits at those barriers and the FMA pipe
// idles a third of the time.  Here
//   * every warp owns a private window (its 256 outputs + the taps' history, filled by its own cp.async copies and
//     ordered by __syncwarp), so nothing about the input is shared between warps;
//   * the one thing the warps of a buffer do share -- the buffer's envelope maximum -- is exchanged split-phase: a warp
//     posts its maximum for buffer t and arrives on an mbarrier, keeps buffer t's 8 outputs per thread in registers,
//     runs the taps of buffer t + 1, and only then waits for buffer t's barrier (long complete), scales and stores.
// Results are bit for bit those of fir_agc_kernel (same tap order, same envelope, same 1 / max).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kSplitTile = 1024;                        // one assembler buffer == one AGC block
constexpr int kSplitPerWarp = kSplitTile / (kFirThreads / 32);

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tma::smem_addr(bar)) : "memory");
}

__global__ void __launch_bounds__(kFirThreads, 5)   // 94 registers; held to 80 for a sixth CTA it spills and is 3 % slower
fir_agc_split_kernel(const float2 *__restrict__ in, long long in_stride, int in_off, float2 *__restrict__ out,
                     long long out_stride, int n_tiles, int kp, float fir_gain, int tiles_per_cta,
                     const __grid_constant__ FirTaps taps)
{
    extern __shared__ __align__(16) float2 xs_all[];   // [warp][2] skewed windows: local i <-> stream sample start - kp + i
    __shared__ __align__(16) float hs[kMaxFirTaps];
    __shared__ float red[2][kFirThreads / 32];
    __shared__ __align__(8) uint64_t bars[2];
    const int c = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int window = kp + kSplitPerWarp;
    const int wlen = fir_window_len(window);
    const int first = blockIdx.x * tiles_per_cta, last = min(first + tiles_per_cta, n_tiles);
    if (first >= last) return;
    for (int k = tid; k < kp; k += kFirThreads) hs[k] = taps.h[k];
    if (tid == 0) {
        tma::mbar_init(&bars[0], kFirThreads / 32);
        tma::mbar_init(&bars[1], kFirThreads / 32);
    }
    __syncthreads();   // taps and barriers: the only block-wide barrier of the kernel
    float2 *xw = xs_all + (size_t)warp * 2 * wlen;
    const float2 *row = in + (size_t)c * in_stride + in_off + warp * kSplitPerWarp - kp;
    float2 *orow = out + (size_t)c * out_stride + warp * kSplitPerWarp + lane * kFirPer;
    // rows, in_off and kp are even: every pair of samples is a 16-byte aligned copy; a lane's copies are 64 samples
    // (80 skewed slots) apart
    auto fill = [&](int blk, float2 *xs) {
        const float2 *s = row + (size_t)blk * kSplitTile + 2 * lane;
        float2 *d = xs + skew8(2 * lane);
        for (int i = 2 * lane; i < window; i += 64, s += 64, d += 80) cp_async16(d, s);
        cp_async_commit();
    };
    const float2 *wfirst = xw + skew8(kp + lane * kFirPer);
    float pi[kFirPer], pq[kFirPer];   // the previous buffer's filtered samples, waiting for its gain
    // the gain of buffer t (local index) once all four warps have posted their maxima, applied to (pi, pq) and stored
    auto finish = [&](int t) {
        const int p = t & 1;
        tma::mbar_wait(&bars[p], (uint32_t)((t >> 1) & 1));
        float m = red[p][0];
#pragma unroll
        for (int wdx = 1; wdx < kFirThreads / 32; wdx++) m = fmaxf(m, red[p][wdx]);
        const float g = __fdiv_rn(1.0f, m);
        float2 *dst = orow + (size_t)(first + t) * kSplitTile;
        if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
            for (int j = 0; j < kFirPer; j += 2)
                *reinterpret_cast<float4 *>(dst + j) = make_float4(__fmul_rn(pi[j], g), __fmul_rn(pq[j], g), __fmul_rn(pi[j + 1], g), __fmul_rn(pq[j + 1], g));
        } else {
#pragma unroll
            for (int j = 0; j < kFirPer; j++) dst[j] = make_float2(__fmul_rn(pi[j], g), __fmul_rn(pq[j], g));
        }
    };
    fill(first, xw);
    for (int blk = first; blk < last; blk++) {
        const int t = blk - first, p = t & 1;
        if (blk + 1 < last) {
            fill(blk + 1, xw + (p ^ 1) * wlen);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncwarp();
        float2 acc[kFirPer];
        fir_taps8(wfirst + p * wlen, hs, kp, acc);
        float ai[kFirPer], aq[kFirPer];
        float m = 0.0001f;
#pragma unroll
        for (int j = 0; j < kFirPer; j++) {
            ai[j] = __fmul_rn(acc[j].x, fir_gain);
            aq[j] = __fmul_rn(acc[j].y, fir_gain);
            const float env = agc_envelope(ai[j], aq[j]);
            if (env > m) m = env;
        }
        // the warp's maximum in one REDUX: m >= 1e-4 and never NaN (a NaN envelope fails `env > m`), and non-negative floats
        // order like their bit patterns
        m = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(m)));
        // the previous buffer first: every warp has read red[p] of buffer t - 2 before it arrives for buffer t - 1, so
        // once that barrier has completed red[p] is free for buffer t
        if (t > 0) finish(t - 1);
        if (lane == 0) {
            red[p][warp] = m;
            mbar_arrive(&bars[p]);
        }
#pragma unroll
        for (int j = 0; j < kFirPer; j++) {
            pi[j] = ai[j];
            pq[j] = aq[j];
        }
        __syncwarp();   // this window is refilled by the warp's own copies two buffers from now
    }
    finish(last - 1 - first);
}

// consecutive tiles of a channel one CTA filters at most, when the bank size chooses (SDRGPU_TUNE_FIR_TILES_PER_CTA
// sets it instead)
constexpr int kFirTilesPerCta = 4;

}  // namespace

namespace sdrgpu {

sdrgpu_status halfband_launch(const float2 *in, long long in_stride, float2 *out, long long out_stride, int out_off,
                              int n_out, int n_channels, const HalfBandTaps &taps, cudaStream_t stream)
{
    dim3 grid((n_out + 255) / 256 > 64 ? 64 : (n_out + 255) / 256, n_channels);
    // the stage's input window starts L - 1 samples before the first new sample
    halfband_kernel<<<grid, 256, 0, stream>>>(in - (taps.length - 1), in_stride, out, out_stride, out_off, n_out, taps);
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    return SDRGPU_OK;
}

sdrgpu_status fir_agc_launch(const FirLaunch &a)
{
    const int kp = fir_padded_taps(a.n_taps);
    // with AGC one CTA == one AGC buffer (the gain is per buffer); otherwise any tiling works
    const int tile = a.agc_block > 0 ? a.agc_block : (a.n < 1024 ? a.n : 1024);
    // double buffer: the next tile's window arrives by cp.async.  While the demodulator of the previous time chunk is
    // running (throttle) the filter is held to a few resident CTAs per SM (sdrgpu_set_tuning)
    const size_t smem_need = sizeof(float2) * 2 * (size_t)fir_window_len(kp + ((tile + 7) & ~7));
    const size_t smem = (a.throttle || g_tuning[SDRGPU_TUNE_THROTTLE_ALWAYS]) ? smem_for_ctas_per_sm(smem_need, sizeof(float) * (kMaxFirTaps + 8), g_tuning[SDRGPU_TUNE_FIR_CTAS_PER_SM]) : smem_need;
    if (smem > 48 * 1024) {
        static size_t fir_attr = 0;
        if (smem > fir_attr) {
            SDRGPU_CUDA(cudaFuncSetAttribute(fir_agc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024 - (int)(sizeof(float) * (kMaxFirTaps + 8))));
            fir_attr = 226 * 1024;
        }
    }
    const int n_tiles = (a.n + tile - 1) / tile;
    // consecutive tiles of a channel per CTA, as long as the grid still fills the GPU a dozen times over
    int tpc = (int)(((long long)a.n_channels * n_tiles) / (148 * 12));
    tpc = tpc < 1 ? 1 : (tpc > kFirTilesPerCta ? kFirTilesPerCta : tpc);
    if (g_tuning[SDRGPU_TUNE_FIR_TILES_PER_CTA] > 0) tpc = g_tuning[SDRGPU_TUNE_FIR_TILES_PER_CTA];
    if (tpc > n_tiles) tpc = n_tiles;
    dim3 grid((n_tiles + tpc - 1) / tpc, a.n_channels);
    // whole 1024-sample AGC buffers (the decoders' framing): per-warp windows and a split-phase exchange of the buffer
    // maximum instead of three block-wide barriers per buffer
    const size_t split_smem = sizeof(float2) * 2 * (kFirThreads / 32) * (size_t)fir_window_len(kp + kSplitPerWarp);
    if (a.agc_block > 0 && tile == kSplitTile && a.n % kSplitTile == 0 && kp >= 8 && smem == smem_need &&
        split_smem <= 48 * 1024 && (a.in_off & 1) == 0) {
        fir_agc_split_kernel<<<grid, kFirThreads, split_smem, a.stream>>>(a.in, a.in_stride, a.in_off, a.out, a.out_stride,
                                                                          n_tiles, kp, a.gain, tpc, *a.taps);
    } else {
        fir_agc_kernel<<<grid, kFirThreads, smem, a.stream>>>(a.in, a.in_stride, a.in_off, a.out, a.out_stride, tile, a.n, kp,
                                                              a.gain, a.agc_block > 0, tpc, *a.taps);
    }
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    return SDRGPU_OK;
}

}  // namespace sdrgpu
