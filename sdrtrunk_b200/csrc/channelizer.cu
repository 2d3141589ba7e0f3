// Polyphase channelizer for sm_100a: 2x-oversampled M-branch filter bank + per-block M-point inverse DFT,
// writing per-channel contiguous streams.
//
// Replaces ComplexPolyphaseChannelizerM2.receive/process + IFFTProcessor
// (J/dsp/filter/channelizer/ComplexPolyphaseChannelizerM2.java:190-235,337-383,407-428) and the strided gather of
// ReusableChannelResultsBuffer.getChannel + gain of OneChannelOutputProcessor.process
// (J/sample/buffer/ReusableChannelResultsBuffer.java:112-153, .../output/OneChannelOutputProcessor.java:81-106).
//
// Math (derived from the reference's aligned filter + top/middle index maps): with M channels, T taps per
// channel, block B (counted from stream start) whose newest complex sample is s_B = (B+1)*M/2 - 1,
//     v_B[n] = sum_{t=0}^{T-1} x[s_B - n - t*M] * h[n + t*M]          n = 0..M-1      (products rounded, added
//                                                                                       in ascending t, no FMA)
//     u_B    = v_B                      (B even, "top" block)
//            = v_B rotated by M/2       (B odd,  "middle" block)
//     out_B[k] = (1/M) * sum_n u_B[n] * e^{+j 2 pi n k / M}
// In units of M/2 samples (unit P = samples [P*M/2, (P+1)*M/2), r = offset inside the unit, n = M/2-1-r):
//     v_B[n]       = sum_t X_P[r] h[n + tM]        with P = B - 2t
//     v_B[n + M/2] = sum_t X_P[r] h[n + M/2 + tM]  with P = B - 1 - 2t
// so one thread that owns r keeps its 2T taps in registers, walks P downwards loading each input sample once
// (coalesced over r) and accumulates NB consecutive blocks in registers.
//
// Data layout in shared memory: [M][NB+1] float2, time index fastest, so every FFT pass (work item =
// butterfly x block) and the final per-channel store (NB consecutive complex samples of one channel = one
// 128-byte line for NB = 16) are bank-conflict free and coalesced.
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <utility>
#include <vector>

#include "common.cuh"
#include "fft_regs.cuh"

using namespace sdrgpu;

namespace {

constexpr int kMaxFactors = 16;
constexpr int kThreads = 256;
constexpr int kMaxEvents = 64;

struct ChanParams {
    const float2 *state;  // [state_len] history ((2T-1)*M/2 samples) followed by the leftover samples
    const float2 *in;     // [n_in] new samples
    const uint8_t *raw;   // pfb2_kernel<..., RAW>: the same samples as 8-bit tuner I/Q (2 bytes per complex sample), converted on load
    int raw_flip, raw_bias;  // value = (int)(byte ^ raw_flip) - raw_bias: signed 8-bit (0x80, 128), unsigned (0, 127)
    const float *taps;    // [M*T] prototype filter h
    const float2 *tw;     // [M] e^{+j 2 pi k / M}
    const float2 *tw2;    // [R1][R2] e^{+j 2 pi n2 k1 / M}: the twiddles between the two steps of pfb2_kernel
    float *out;
    const int *sel;       // [n_sel] bin of each output row (channel layout)
    const float *gain_f;  // [n_sel] float gain (used when gain_exact)
    const double *gain_d; // [n_sel]
    long long out_stride; // floats per output row (channel layout)
    float *out2;          // rows >= n_main (second bins of two-bin channels) go here
    long long out2_stride;
    int n_main;
    int state_len, n_in;
    int M, T, half, H;
    int n_blocks, parity0;
    int n_sel, layout, gain_exact;
    int prefetch_blocks; // L2 read-ahead distance of pfb2_kernel in blocks
    int identity;        // selection is every bin in order with one float-representable gain (gain_uniform)
    float gain_uniform;
    float inv_m;
    int n_factors;
    int factors[kMaxFactors];
    unsigned magic_s[kMaxFactors];  // ceil(2^32 / s) for the stride of each pass
    // pfb2_kernel, every bin a frequency-corrected one-bin channel (OneChannelOutputProcessor + Oscillator) with one
    // float-representable gain: mixed where step B stores the rows.  osc = the look-ahead rings [M][osc_ring_len]
    // (osc_produce_kernel; row == bin == oscillator), osc_start = ring slot of this call's first block; else nullptr
    const float2 *osc;
    int osc_ring_len, osc_start;
    float2 *next_state;  // pfb2_kernel only: one CTA also writes the next call's history (else save_state_kernel)
    int next_len, consumed;
    float neg_zero;      // -0.0f as a run-time value: the addend of the filter bank's packed products (fb_thread)
};

// ByteSampleConverter / SignedByteSampleConverter (J/source/tuner/... lookup tables: (b - 127) / 128.0f, b / 128.0f): both
// steps are exact in float, so converting on load gives the bits convert_kernel would have written
__device__ __forceinline__ float2 load_raw(const ChanParams &p, long long idx)
{
    const uchar2 b = __ldg(reinterpret_cast<const uchar2 *>(p.raw) + idx);
    const int vi = (int)(b.x ^ p.raw_flip) - p.raw_bias, vq = (int)(b.y ^ p.raw_flip) - p.raw_bias;
    return make_float2(__fmul_rn((float)vi, 0.0078125f), __fmul_rn((float)vq, 0.0078125f));
}

template <bool RAW = false>
__device__ __forceinline__ float2 load_x(const ChanParams &p, int unit, int r)
{
    // virtual concatenation [state | in | zeros]; unit 0 starts right after the history
    int idx = p.H + unit * p.half + r;
    if (idx < p.state_len) return __ldg(p.state + idx);
    idx -= p.state_len;
    if (idx < p.n_in) return RAW ? load_raw(p, idx) : __ldg(p.in + idx);
    return make_float2(0.0f, 0.0f);
}

__device__ __forceinline__ float2 cmul(float2 a, float2 w)
{
    // explicit FMA is fine here: the inverse DFT is compared at 1e-4 relative RMS, not bit-exactly
    return make_float2(fmaf(a.x, w.x, -a.y * w.y), fmaf(a.x, w.y, a.y * w.x));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 jmul(float2 a) { return make_float2(-a.y, a.x); }  // * (+j)

template <int NB, int TT>
__global__ void __launch_bounds__(kThreads) pfb_ifft_kernel(const ChanParams p)
{
    extern __shared__ float2 smem[];
    constexpr int LD = NB + 1;
    const int M = p.M, half = p.half;
    float2 *buf0 = smem;
    float2 *buf1 = smem + (size_t)M * LD;
    float2 *tw = smem + 2 * (size_t)M * LD;
    const int tid = threadIdx.x;
    const int b0 = blockIdx.x * NB;

    for (int i = tid; i < M; i += kThreads) tw[i] = p.tw[i];

    // ------------------------------------------------------------------ filter bank
    for (int r = tid; r < half; r += kThreads) {
        const int n = half - 1 - r;
        if constexpr (TT > 0) {
            float hA[TT], hB[TT];
#pragma unroll
            for (int t = 0; t < TT; t++) {
                hA[t] = __ldg(p.taps + n + t * M);
                hB[t] = __ldg(p.taps + n + half + t * M);
            }
            float2 accA[NB], accB[NB];
#pragma unroll
            for (int pp = NB - 1; pp >= -(2 * TT - 1); --pp) {
                const float2 x = load_x(p, b0 + pp, r);
#pragma unroll
                for (int t = 0; t < TT; t++) {
                    const int bl = pp + 2 * t;  // branch n: unit P = B - 2t
                    if (bl >= 0 && bl < NB) {
                        const float px = __fmul_rn(x.x, hA[t]), py = __fmul_rn(x.y, hA[t]);
                        if (t == 0) accA[bl] = make_float2(__fadd_rn(0.0f, px), __fadd_rn(0.0f, py));
                        else accA[bl] = make_float2(__fadd_rn(accA[bl].x, px), __fadd_rn(accA[bl].y, py));
                    }
                    const int bm = pp + 1 + 2 * t;  // branch n + M/2: unit P = B - 1 - 2t
                    if (bm >= 0 && bm < NB) {
                        const float px = __fmul_rn(x.x, hB[t]), py = __fmul_rn(x.y, hB[t]);
                        if (t == 0) accB[bm] = make_float2(__fadd_rn(0.0f, px), __fadd_rn(0.0f, py));
                        else accB[bm] = make_float2(__fadd_rn(accB[bm].x, px), __fadd_rn(accB[bm].y, py));
                    }
                }
            }
#pragma unroll
            for (int bl = 0; bl < NB; bl++) {
                const int odd = (p.parity0 + b0 + bl) & 1;
                buf0[(size_t)(odd ? n + half : n) * LD + bl] = accA[bl];
                buf0[(size_t)(odd ? n : n + half) * LD + bl] = accB[bl];
            }
        } else {
            for (int bl = 0; bl < NB; bl++) {
                float2 a = make_float2(0.0f, 0.0f), b = make_float2(0.0f, 0.0f);
                for (int t = 0; t < p.T; t++) {
                    const float ha = __ldg(p.taps + n + t * M), hb = __ldg(p.taps + n + half + t * M);
                    const float2 xa = load_x(p, b0 + bl - 2 * t, r);
                    const float2 xb = load_x(p, b0 + bl - 1 - 2 * t, r);
                    a = make_float2(__fadd_rn(a.x, __fmul_rn(xa.x, ha)), __fadd_rn(a.y, __fmul_rn(xa.y, ha)));
                    b = make_float2(__fadd_rn(b.x, __fmul_rn(xb.x, hb)), __fadd_rn(b.y, __fmul_rn(xb.y, hb)));
                }
                const int odd = (p.parity0 + b0 + bl) & 1;
                buf0[(size_t)(odd ? n + half : n) * LD + bl] = a;
                buf0[(size_t)(odd ? n : n + half) * LD + bl] = b;
            }
        }
    }
    __syncthreads();

    // ------------------------------------------------------------------ inverse DFT: Stockham autosort passes,
    // decimation in frequency:  y[q + s(r p + k)] = (sum_j x[q + s(p + m j)] W_r^{jk}) * w_M^{s p k}
    float2 *src = buf0, *dst = buf1;
    int s = 1;
    for (int f = 0; f < p.n_factors; f++) {
        const int r = p.factors[f];
        const int m = M / (r * s);
        const int items = (M / r) * NB;
        const unsigned magic = p.magic_s[f];
        for (int item = tid; item < items; item += kThreads) {
            const int bl = item % NB;
            const int bf = item / NB;
            const int pq = (s == 1) ? bf : (int)__umulhi((unsigned)bf, magic);
            const int q = bf - pq * s;
            const float2 *x = src + (size_t)(q + s * pq) * LD + bl;
            float2 *y = dst + (size_t)(q + s * r * pq) * LD + bl;
            const size_t xs = (size_t)s * m * LD;  // input stride between j
            const size_t ys = (size_t)s * LD;      // output stride between k
            const int tws = s * pq;                // twiddle index step
            if (r == 4) {
                const float2 a = x[0], b = x[xs], c = x[2 * xs], d = x[3 * xs];
                const float2 t0 = cadd(a, c), t1 = csub(a, c), t2 = cadd(b, d), t3 = jmul(csub(b, d));
                y[0] = cadd(t0, t2);
                y[ys] = cmul(cadd(t1, t3), tw[tws]);
                y[2 * ys] = cmul(csub(t0, t2), tw[2 * tws]);
                y[3 * ys] = cmul(csub(t1, t3), tw[3 * tws]);
            } else if (r == 2) {
                const float2 a = x[0], b = x[xs];
                y[0] = cadd(a, b);
                y[ys] = cmul(csub(a, b), tw[tws]);
            } else if (r == 5) {
                const float c1 = 0.30901699437494742f, c2 = -0.80901699437494742f;
                const float s1 = 0.95105651629515357f, s2 = 0.58778525229247313f;
                const float2 a = x[0], b = x[xs], c = x[2 * xs], d = x[3 * xs], e = x[4 * xs];
                const float2 t1 = cadd(b, e), t2 = cadd(c, d), t3 = csub(b, e), t4 = csub(c, d);
                const float2 m1 = make_float2(a.x + c1 * t1.x + c2 * t2.x, a.y + c1 * t1.y + c2 * t2.y);
                const float2 m2 = make_float2(a.x + c2 * t1.x + c1 * t2.x, a.y + c2 * t1.y + c1 * t2.y);
                const float2 n1 = jmul(make_float2(s1 * t3.x + s2 * t4.x, s1 * t3.y + s2 * t4.y));
                const float2 n2 = jmul(make_float2(s2 * t3.x - s1 * t4.x, s2 * t3.y - s1 * t4.y));
                y[0] = make_float2(a.x + t1.x + t2.x, a.y + t1.y + t2.y);
                y[ys] = cmul(cadd(m1, n1), tw[tws]);
                y[2 * ys] = cmul(cadd(m2, n2), tw[2 * tws]);
                y[3 * ys] = cmul(csub(m2, n2), tw[3 * tws]);
                y[4 * ys] = cmul(csub(m1, n1), tw[4 * tws]);
            } else if (r == 3) {
                const float sq = 0.86602540378443865f;
                const float2 a = x[0], b = x[xs], c = x[2 * xs];
                const float2 t = cadd(b, c), u = jmul(csub(b, c));
                const float2 mm = make_float2(a.x - 0.5f * t.x, a.y - 0.5f * t.y);
                const float2 nn = make_float2(sq * u.x, sq * u.y);
                y[0] = cadd(a, t);
                y[ys] = cmul(cadd(mm, nn), tw[tws]);
                y[2 * ys] = cmul(csub(mm, nn), tw[2 * tws]);
            } else {
                // generic prime radix: direct r x r DFT from the M-th root table
                const int step = M / r;
                for (int k = 0; k < r; k++) {
                    float2 acc = make_float2(0.0f, 0.0f);
                    int widx = 0;
                    for (int j = 0; j < r; j++) {
                        acc = cadd(acc, cmul(x[j * xs], tw[widx]));
                        widx += k * step;
                        if (widx >= M) widx %= M;
                    }
                    y[k * ys] = cmul(acc, tw[tws * k]);
                }
            }
        }
        __syncthreads();
        float2 *tmp = src;
        src = dst;
        dst = tmp;
        s *= r;
    }

    // ------------------------------------------------------------------ scale + store
    const float inv_m = p.inv_m;
    if (p.layout == SDRGPU_LAYOUT_CHANNELS) {
        const int total = p.n_sel * NB;
        for (int i = tid; i < total; i += kThreads) {
            const int bl = i % NB, c = i / NB;
            const int b = b0 + bl;
            if (b >= p.n_blocks) continue;
            float2 v = src[(size_t)__ldg(p.sel + c) * LD + bl];
            v.x = __fmul_rn(v.x, inv_m);  // FloatFFT_1D.complexInverse(a, true): a[i] *= 1.0f / n
            v.y = __fmul_rn(v.y, inv_m);
            if (p.gain_exact) {  // float * float == (float)(float * double) when the gain is float-representable
                const float g = __ldg(p.gain_f + c);
                v.x = __fmul_rn(v.x, g);
                v.y = __fmul_rn(v.y, g);
            } else {  // ReusableComplexBuffer.applyGain: samples[x] *= (double)gain
                const double g = __ldg(p.gain_d + c);
                v.x = __double2float_rn(__dmul_rn((double)v.x, g));
                v.y = __double2float_rn(__dmul_rn((double)v.y, g));
            }
            float *row = c < p.n_main ? p.out + (size_t)c * p.out_stride : p.out2 + (size_t)(c - p.n_main) * p.out2_stride;
            *reinterpret_cast<float2 *>(row + 2 * (size_t)b) = v;
        }
    } else {
        const int total = M * NB;
        for (int i = tid; i < total; i += kThreads) {
            const int k = i % M, bl = i / M;
            const int b = b0 + bl;
            if (b >= p.n_blocks) continue;
            float2 v = src[(size_t)k * LD + bl];
            v.x = __fmul_rn(v.x, inv_m);
            v.y = __fmul_rn(v.y, inv_m);
            *reinterpret_cast<float2 *>(p.out + ((size_t)b * M + k) * 2) = v;
        }
    }
}


// ---------------------------------------------------------------------------------------------------------------
// pfb2_kernel: the fast path for channel counts that split as M = R1 * R2 with register-sized factors
// (400 = 20 x 20, 800 = 32 x 25, 96 = 8 x 12, ... see sdrgpu_chan_create).  One CTA per tile of NB consecutive blocks:
//   0. L2 read-ahead of the input the tile one wave later will need (its first touch is otherwise a DRAM round trip)
//   1. filter bank (as above: thread <-> input offset r, taps in registers, NB blocks of two branches accumulated
//      in registers, products rounded and added in tap order like the Java)         -> V[b][n]         (shared)
//   2. step A: thread (b, n2) runs an R1-point DFT over n1 of V[b][R2 n1 + n2] in registers, multiplies by
//      W_M^{n2 k1}                                                                  -> Y[b][k1][n2]    (shared)
//      (NB = 8: V is stored in Y's layout and step A transforms it in place -- see Pfb2Layout)
//   3. step B: thread (b, k1) runs an R2-point DFT over n2 in registers: bin k1 + R1 k2.  With the default selection
//      (every bin, one gain) and NB = 8 the 8 lanes holding one bin's 8 consecutive samples scale and write them
//      straight to the channel's row (64 contiguous bytes) -- done.  Otherwise                -> X[b][k] (shared)
//   4. (general selection) rows of NB consecutive samples per selected channel -> HBM, scaled by 1/M and the gain
// Shared-memory traffic is 4 passes over the tile (6 with step 4) instead of 10 for the radix-4/5 Stockham version,
// all bank-conflict free (Pfb2Layout), and the index arithmetic is compile-time.
// ---------------------------------------------------------------------------------------------------------------
template <int R2>
struct YPad {
    static constexpr int even = (R2 + 1) & ~1;
    static constexpr int value = ((even / 2) & 1) ? even : even + 2;   // float2 per (b, k1) row
};

template <int M, int R1, int R2, int NB, int TT, int NT>
struct Pfb2Layout {
    static_assert(NB == 8 || NB == 16, "strides and thread mappings are chosen for 8 or 16 blocks per tile");
    static constexpr int Mp = (M + 15) & ~15;
    // NB == 8: steps A and B map lanes to (block fastest, then n2 / k1): 8 lanes of one n2 / k1 and their neighbour
    // form a half-warp, so every per-block row stride == 2 (mod 16 float2) spreads a half-warp over all 16 banks --
    // V reads, Y writes, Y LDS.128 reads (stride / 2 odd), X writes and the store pass's X reads are all conflict free.
    // NB == 16 (small M): lanes run over n2 / k1 first; strides == 4 (mod 16) keep row-straddling half-warps apart.
    static constexpr int SV = NB == 8 ? Mp + 2 : Mp + 4;      // V[b][n]
    static constexpr int XS = NB == 8 ? Mp + 2 : Mp + 1;      // X[b][k]
    static constexpr int R2P = YPad<R2>::value;               // Y[b][k1][R2P]
    static constexpr int y_base = R1 * R2P;
    static constexpr int y_want = NB == 8 ? 2 : (((R2 % 16) + 1) & ~1);
    static constexpr int YB = y_base + ((y_want - y_base % 16) + 16) % 16;
    // NB == 8: the filter bank writes V[b][R2 n1 + n2] straight into Y's layout, at Y[b][n1][n2].  Step A's thread (b, n2)
    // reads column n2 of block b for every n1 and writes the same column for every k1, so it transforms in place and V
    // needs no region of its own; X (general selection) gets one behind Y.  NB == 16: V / X share region 0, Y follows.
    static constexpr bool v_in_y = NB == 8;
    static constexpr int region0 = v_in_y ? NB * XS : (NB * SV > NB * XS) ? NB * SV : NB * XS;
    static constexpr int y_off = v_in_y ? 0 : region0, x_off = v_in_y ? NB * YB : 0;
    static constexpr size_t smem_bytes = sizeof(float2) * (size_t)(region0 + NB * YB);
    static constexpr size_t smem_direct = v_in_y ? sizeof(float2) * (size_t)(NB * YB) : smem_bytes;   // no X
};

// V[bl * SV + vidx(n)]: vidx(n) = n, or with R2 > 0 the row layout of Y, R2 = row length, R2P = row pitch
template <int M, int NB, int TT, bool FAST, bool RAW, int R2 = 0, int R2P = 0>
__device__ __forceinline__ void fb_thread(const ChanParams &p, const float2 *__restrict__ xin, long long first, int b0, int r,
                                          float2 *V, int SV)
{
    constexpr int half = M / 2;
    const int n = half - 1 - r;
    float hA[TT], hB[TT];
#pragma unroll
    for (int t = 0; t < TT; t++) {
        hA[t] = __ldg(p.taps + n + t * M);
        hB[t] = __ldg(p.taps + n + half + t * M);
    }
    float2 accA[NB], accB[NB];
    // The Java rounds the product and the sum separately (no Math.fma in the filter bank).  The I and Q rails share packed
    // instructions: the product is an FFMA2 whose addend is -0.0 (x h + -0 is the rounded product, signed zeros included),
    // the sum an FADD2 -- two instructions where four scalar ones were.  The -0.0 is a kernel parameter on purpose: ptxas
    // contracts mul.rn.f32x2 + add.rn.f32x2, and an FFMA2 with a literal -0.0 addend + add, into ONE FFMA2 whatever -fmad
    // says (checked in the SASS; round 1 gave the packed filter bank up for that reason).
    const float2 nz = make_float2(p.neg_zero, p.neg_zero);
#pragma unroll
    for (int pp = NB - 1; pp >= -(2 * TT - 1); --pp) {
        const float2 x = !FAST ? load_x<RAW>(p, b0 + pp, r)
                         : (RAW ? load_raw(p, first + (pp + 2 * TT - 1) * half + r) : __ldg(xin + (pp + 2 * TT - 1) * half + r));
#pragma unroll
        for (int t = 0; t < TT; t++) {
            const int bl = pp + 2 * t;  // branch n: unit P = B - 2t
            if (bl >= 0 && bl < NB) {
#ifdef SDRGPU_PFB_FMA
                if (t == 0) accA[bl] = make_float2(__fmul_rn(x.x, hA[t]), __fmul_rn(x.y, hA[t]));
                else accA[bl] = make_float2(__fmaf_rn(x.x, hA[t], accA[bl].x), __fmaf_rn(x.y, hA[t], accA[bl].y));
#else
                const float2 pr = __ffma2_rn(x, make_float2(hA[t], hA[t]), nz);
                // (the Java's 0.0f + product differs from the product only in the sign of a zero)
                if (t == 0) accA[bl] = pr;
                else accA[bl] = __fadd2_rn(accA[bl], pr);
#endif
            }
            const int bm = pp + 1 + 2 * t;  // branch n + M/2: unit P = B - 1 - 2t
            if (bm >= 0 && bm < NB) {
#ifdef SDRGPU_PFB_FMA
                if (t == 0) accB[bm] = make_float2(__fmul_rn(x.x, hB[t]), __fmul_rn(x.y, hB[t]));
                else accB[bm] = make_float2(__fmaf_rn(x.x, hB[t], accB[bm].x), __fmaf_rn(x.y, hB[t], accB[bm].y));
#else
                const float2 pr = __ffma2_rn(x, make_float2(hB[t], hB[t]), nz);
                if (t == 0) accB[bm] = pr;
                else accB[bm] = __fadd2_rn(accB[bm], pr);
#endif
            }
        }
    }
    const int par = (p.parity0 + b0) & 1;
    const int ilo = R2 > 0 ? (n / R2) * R2P + n % R2 : n;
    const int ihi = R2 > 0 ? ((n + half) / R2) * R2P + (n + half) % R2 : n + half;
#pragma unroll
    for (int bl = 0; bl < NB; bl++) {
        const int odd = (par + bl) & 1;   // "middle" blocks: the two halves swap (the M/2 circular shift)
        V[bl * SV + (odd ? ihi : ilo)] = accA[bl];
        V[bl * SV + (odd ? ilo : ihi)] = accB[bl];
    }
}

template <int M, int R1, int R2, int NB, int TT, int NT, int MINB, bool RAW>
// M = 800 runs three CTAs per SM: 80 registers (no spill; 8 bytes with 8-bit input) and, with V inside Y, 53 KB of shared
// memory per CTA on the direct-store path.  The third CTA's phases fill the barriers of the other two: 1.40 -> 1.15 ms per
// 8 launches on a B200 at 1000 W (profiles/r5f_pfb_pipe_time.txt); 3 x 256 x 80 registers still leave 4 K to the one-warp oscillator
// producers of frequency-corrected channels.  M = 400 needs its 72 (64: a spill, 1 % slower).
__global__ void __launch_bounds__(NT, MINB) pfb2_kernel(const ChanParams p)
{
    using L = Pfb2Layout<M, R1, R2, NB, TT, NT>;
    constexpr int half = M / 2, SV = L::SV, XS = L::XS, R2P = L::R2P, YB = L::YB;
    extern __shared__ __align__(16) float2 smem[];
    float2 *Y = smem + L::y_off;      // [NB][R1][R2P]
    float2 *V = L::v_in_y ? Y : smem; // [NB][SV], or Y's layout
    float2 *X = smem + L::x_off;      // [NB][XS]
    constexpr int VS = L::v_in_y ? YB : SV, VR2 = L::v_in_y ? R2 : 0, VR2P = L::v_in_y ? R2P : 0;
    const int tid = threadIdx.x;
    const int b0 = blockIdx.x * NB;

    // the history the next call starts from, next_state[i] = [state | in][consumed + i]: a few KB copied by one CTA of
    // the middle of the grid into the other half of the state ping-pong (a separate launch costs 3 % of the step)
    if (p.next_state != nullptr && blockIdx.x == (gridDim.x >> 1)) {
        for (int i = tid; i < p.next_len; i += NT) {
            const int idx = p.consumed + i;
            float2 v = make_float2(0.0f, 0.0f);
            if (idx < p.state_len) v = p.state[idx];
            else if (idx - p.state_len < p.n_in) v = RAW ? load_raw(p, idx - p.state_len) : p.in[idx - p.state_len];
            p.next_state[i] = v;
        }
    }

    // ------------------------------------------------------------------ 1. filter bank
    {
        // every sample this tile needs lies in the new input (true for all but the first tiles of a call)
        const long long first = (long long)b0 * half - p.state_len;                    // index into p.in of unit b0-(2T-1)
        const bool fast = first >= 0 && first + (long long)(NB + 2 * TT - 1) * half <= p.n_in;
        const float2 *xin = RAW ? nullptr : p.in + (fast ? first : 0);
        {
            // pull the new input of the tile that will run about a wave later into L2: the first touch of every input
            // line otherwise costs the filter bank a DRAM round trip (+10 % measured)
            const long long ahead = first + (long long)(2 * TT - 1 + (long long)p.prefetch_blocks) * half;
            const int lines = NB * half * (RAW ? 2 : (int)sizeof(float2)) / 128;
            if (ahead >= 0 && ahead + (long long)NB * half <= p.n_in)
                for (int i = tid; i < lines; i += NT) {
                    if (RAW) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.raw + 2 * ahead + i * 128));
                    else asm volatile("prefetch.global.L2 [%0];" ::"l"(p.in + ahead + i * 16));
                }
        }
        if (fast) {
            for (int r = tid; r < half; r += NT) fb_thread<M, NB, TT, true, RAW, VR2, VR2P>(p, xin, first, b0, r, V, VS);
        } else {
            for (int r = tid; r < half; r += NT) fb_thread<M, NB, TT, false, RAW, VR2, VR2P>(p, xin, first, b0, r, V, VS);
        }
    }
    __syncthreads();

    // ------------------------------------------------------------------ 2. step A: R1-point DFTs over n1
    for (int item = tid; item < NB * R2; item += NT) {
        const int b = NB == 8 ? (item & 7) : item / R2, n2 = NB == 8 ? (item >> 3) : item - b * R2;
        float2 a[R1];
        const float2 *v = V + b * VS + n2;
#pragma unroll
        for (int n1 = 0; n1 < R1; n1++) a[n1] = v[(L::v_in_y ? R2P : R2) * n1];
        rfft::dft<R1>(a);
        float2 *y = Y + b * YB + n2;
        y[0] = a[0];
#pragma unroll
        for (int k1 = 1; k1 < R1; k1++) {
            const float2 w = __ldg(p.tw2 + k1 * R2 + n2);
            y[k1 * R2P] = rfft::cmul(a[k1], w.x, w.y);
        }
    }
    __syncthreads();

    // ------------------------------------------------------------------ 3. step B: R2-point DFTs over n2
    // Default selection (every bin in order, one float-representable gain) with block-fastest lanes: the 8 lanes that
    // hold one bin's 8 consecutive samples write them straight to that channel's row (64 contiguous bytes), so the
    // X transpose, its barrier and the store pass are skipped.
    const bool direct = NB == 8 && p.identity && p.layout == SDRGPU_LAYOUT_CHANNELS;
    for (int item = tid; item < NB * R1; item += NT) {
        const int b = NB == 8 ? (item & 7) : item / R1, k1 = NB == 8 ? (item >> 3) : item - b * R1;
        float2 a[R2];
        const float4 *y = reinterpret_cast<const float4 *>(Y + b * YB + k1 * R2P);
#pragma unroll
        for (int i = 0; i < R2 / 2; i++) {
            const float4 v = y[i];
            a[2 * i] = make_float2(v.x, v.y);
            a[2 * i + 1] = make_float2(v.z, v.w);
        }
        if (R2 & 1) a[R2 - 1] = Y[b * YB + k1 * R2P + R2 - 1];
        rfft::dft<R2>(a);
        if (direct) {
            if (b0 + b < p.n_blocks) {
                // FloatFFT_1D.complexInverse(a, true): a[i] *= 1.0f / n; then applyGain
                const float inv = p.inv_m, g = p.gain_uniform;
                float *o = p.out + (size_t)k1 * p.out_stride + 2 * (size_t)(b0 + b);
                const size_t ostep = (size_t)R1 * p.out_stride;
                if (p.osc != nullptr) {
                    // every bin frequency-corrected (OneChannelOutputProcessor + Oscillator, row == bin == oscillator): the
                    // oscillator value of this block from the look-ahead rings, multiplied in between the 1/M of the inverse
                    // FFT and the gain -- the arithmetic of osc_mix_kernel on the value it would have read back
                    int slot = p.osc_start + b0 + b;
                    if (slot >= p.osc_ring_len) slot -= p.osc_ring_len;
                    const float2 *zp = p.osc + (size_t)k1 * p.osc_ring_len + slot;
                    const size_t zstep = (size_t)R1 * p.osc_ring_len;
#pragma unroll
                    for (int k2 = 0; k2 < R2; k2++) {
                        const float2 z = __ldg(zp);
                        const float vx = __fmul_rn(a[k2].x, inv), vy = __fmul_rn(a[k2].y, inv);
                        float2 v;
                        v.x = __fmul_rn(__fsub_rn(__fmul_rn(vx, z.x), __fmul_rn(vy, z.y)), g);
                        v.y = __fmul_rn(__fadd_rn(__fmul_rn(vy, z.x), __fmul_rn(vx, z.y)), g);
                        *reinterpret_cast<float2 *>(o) = v;
                        o += ostep;
                        zp += zstep;
                    }
                } else {
#pragma unroll
                    for (int k2 = 0; k2 < R2; k2++) {
                        // (1 / M, then the gain: two packed multiplies for four scalar ones)
                        const float2 v = __fmul2_rn(__fmul2_rn(a[k2], make_float2(inv, inv)), make_float2(g, g));
                        *reinterpret_cast<float2 *>(o) = v;
                        o += ostep;
                    }
                }
            }
        } else {
            float2 *xo = X + b * XS + k1;
#pragma unroll
            for (int k2 = 0; k2 < R2; k2++) xo[R1 * k2] = a[k2];
        }
    }
    if (direct) return;
    __syncthreads();

    // ------------------------------------------------------------------ 4. scale + store
    // FloatFFT_1D.complexInverse(a, true): a[i] *= 1.0f / n; then ReusableComplexBuffer.applyGain: samples[x] *= gain
    // (a double; float * float == (float)(float * double) when the gain is float-representable: gain_exact)
    const float inv_m = p.inv_m;
    if (p.layout == SDRGPU_LAYOUT_CHANNELS) {
        // NB consecutive lanes write the NB consecutive samples of one channel row (128 bytes for NB = 16)
        constexpr int ROWS = NT / NB;                  // channel rows per pass over the CTA
        const int bl = tid % NB, row0 = tid / NB;
        const int b = b0 + bl;
        if (tid < ROWS * NB && b < p.n_blocks) {
            float *out = p.out + 2 * (size_t)b;
            if (p.identity) {
                // default selection: every bin in order, one float-representable gain
                const float g = p.gain_uniform;
                float *o = out + (size_t)row0 * p.out_stride;
                const size_t ostep = (size_t)ROWS * p.out_stride;
                const float2 *xr = X + bl * XS;
#pragma unroll 5
                for (int c = row0; c < M; c += ROWS) {
                    float2 v = xr[c];
                    v.x = __fmul_rn(__fmul_rn(v.x, inv_m), g);
                    v.y = __fmul_rn(__fmul_rn(v.y, inv_m), g);
                    *reinterpret_cast<float2 *>(o) = v;
                    o += ostep;
                }
            } else if (p.gain_exact) {
                for (int c = row0; c < p.n_sel; c += ROWS) {
                    const float g = __ldg(p.gain_f + c);
                    float2 v = X[bl * XS + __ldg(p.sel + c)];
                    v.x = __fmul_rn(__fmul_rn(v.x, inv_m), g);
                    v.y = __fmul_rn(__fmul_rn(v.y, inv_m), g);
                    float *row = c < p.n_main ? p.out + (size_t)c * p.out_stride : p.out2 + (size_t)(c - p.n_main) * p.out2_stride;
                    *reinterpret_cast<float2 *>(row + 2 * (size_t)b) = v;
                }
            } else {
                for (int c = row0; c < p.n_sel; c += ROWS) {
                    const double g = __ldg(p.gain_d + c);
                    float2 v = X[bl * XS + __ldg(p.sel + c)];
                    v.x = __double2float_rn(__dmul_rn((double)__fmul_rn(v.x, inv_m), g));
                    v.y = __double2float_rn(__dmul_rn((double)__fmul_rn(v.y, inv_m), g));
                    float *row = c < p.n_main ? p.out + (size_t)c * p.out_stride : p.out2 + (size_t)(c - p.n_main) * p.out2_stride;
                    *reinterpret_cast<float2 *>(row + 2 * (size_t)b) = v;
                }
            }
        }
    } else {
        const int total = M * NB;
        for (int i = tid; i < total; i += NT) {
            const int k = i % M, bl = i / M;
            const int b = b0 + bl;
            if (b >= p.n_blocks) continue;
            float2 v = X[bl * XS + k];
            v.x = __fmul_rn(v.x, inv_m);
            v.y = __fmul_rn(v.y, inv_m);
            *reinterpret_cast<float2 *>(p.out + ((size_t)b * M + k) * 2) = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Post-processing of the "special" output channels, in place on their rows, one warp per channel:
//   two-bin channels  TwoChannelOutputProcessor.process + TwoChannelSynthesizerM2.process + FS4DownConverter
//                     (J/dsp/filter/channelizer/output/TwoChannelOutputProcessor.java:98-121,
//                      J/dsp/filter/channelizer/TwoChannelSynthesizerM2.java:90-158, J/dsp/mixer/FS4DownConverter.java:32-68)
//   frequency offset  Oscillator mix (J/dsp/mixer/Oscillator.java:42-68, AbstractOscillator.java:102-116): the rotator
//                     is a float recursion with fastNormalize, so it runs as a sequential chain that every lane
//                     walks, lane i keeping the value of sample i
//   gain              ReusableComplexBuffer.applyGain: samples[x] = (float)(samples[x] * (double) gain)
// The pfb kernels leave these rows at gain 1 (bin values after the 1/M of the inverse FFT).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kMaxSynthEntries = 32;   // serpentine entries (4 floats each): filter.length / 2

struct PostChannel {
    int row, row2;          // output row; scratch row of the second bin (-1 for one-bin channels)
    int mix;                // oscillator enabled
    float angle_i, angle_q; // Oscillator: Complex.fromAngle((float)(2 pi f / fs))
    double gain;
};

struct PostState {
    float cur_i, cur_q;     // Oscillator current vector, starts at (0, -1)
    int top_block, fs4;
    float4 hist[kMaxSynthEntries];  // the newest serpentine entries, oldest first
};

struct SynthFilter {
    float f[4 * kMaxSynthEntries];  // taps duplicated for I and Q (TwoChannelSynthesizerM2.init)
    int entries;                     // len / 4
};

__global__ void __launch_bounds__(32) post_channel_kernel(float *out, long long out_stride, const float *out2,
                                                          long long out2_stride, int n, const PostChannel *chans,
                                                          PostState *states, const __grid_constant__ SynthFilter filt)
{
    __shared__ float4 ent[kMaxSynthEntries + 32];
    const int lane = threadIdx.x;
    const PostChannel c = chans[blockIdx.x];
    PostState *st = states + blockIdx.x;
    float2 *row = reinterpret_cast<float2 *>(out + (size_t)c.row * out_stride);
    const float2 *row2 = c.row2 >= 0 ? reinterpret_cast<const float2 *>(out2 + (size_t)c.row2 * out2_stride) : nullptr;
    const int H = filt.entries - 1;   // history entries a sample needs besides its own
    float cur_i = st->cur_i, cur_q = st->cur_q;
    const int top0 = st->top_block, fs40 = st->fs4;
    if (row2)
        for (int i = lane; i < H; i += 32) ent[i] = st->hist[i];
    __syncwarp();
    for (int base = 0; base < n; base += 32) {
        const int k = base + lane;
        const bool valid = k < n;
        float2 v = valid ? row[k] : make_float2(0.f, 0.f);
        if (row2) {
            const float2 b = valid ? row2[k] : make_float2(0.f, 0.f);
            // FloatFFT_1D(2).complexInverse(buffer, true): butterfly, then * 1/2
            const float i0 = __fmul_rn(__fadd_rn(v.x, b.x), 0.5f), i1 = __fmul_rn(__fadd_rn(v.y, b.y), 0.5f);
            const float i2 = __fmul_rn(__fsub_rn(v.x, b.x), 0.5f), i3 = __fmul_rn(__fsub_rn(v.y, b.y), 0.5f);
            const bool top = ((top0 ^ k) & 1) != 0;   // mTopBlockIndicator toggles per sample
            ent[H + lane] = top ? make_float4(i0, i1, i2, i3) : make_float4(i2, i3, i0, i1);
            __syncwarp();
            // product[y] = serpentine[y] * filter[y]; accumulators sum the I / Q lanes in index order
            float acc_i = 0.0f, acc_q = 0.0f;
            for (int j = 0; j < filt.entries; j++) {
                const float4 e = ent[H + lane - j];
                const float p0 = __fmul_rn(e.x, filt.f[4 * j]), p1 = __fmul_rn(e.y, filt.f[4 * j + 1]);
                const float p2 = __fmul_rn(e.z, filt.f[4 * j + 2]), p3 = __fmul_rn(e.w, filt.f[4 * j + 3]);
                acc_i = __fadd_rn(__fadd_rn(acc_i, p0), p2);
                acc_q = __fadd_rn(__fadd_rn(acc_q, p1), p3);
            }
            // FS4DownConverter: multiply by (-j)^pointer
            switch ((fs40 + k) & 3) {
                case 1: v = make_float2(acc_q, -acc_i); break;
                case 2: v = make_float2(-acc_i, -acc_q); break;
                case 3: v = make_float2(-acc_q, acc_i); break;
                default: v = make_float2(acc_i, acc_q); break;
            }
            __syncwarp();
            // keep the newest H entries for the next 32 samples
            const int count = min(32, n - base);
            float4 keep = make_float4(0.f, 0.f, 0.f, 0.f);
            if (lane < H) keep = ent[count + lane];
            __syncwarp();
            if (lane < H) ent[lane] = keep;
            __syncwarp();
        }
        if (c.mix) {
            // AbstractOscillator.mixComplex: sample * current, then rotate(): current *= angle, fastNormalize
            float my_i = cur_i, my_q = cur_q;
            const int count = min(32, n - base);
            for (int i = 0; i < count; i++) {
                if (i == lane) {
                    my_i = cur_i;
                    my_q = cur_q;
                }
                const float ni = __fsub_rn(__fmul_rn(cur_i, c.angle_i), __fmul_rn(cur_q, c.angle_q));
                const float nq = __fadd_rn(__fmul_rn(cur_q, c.angle_i), __fmul_rn(cur_i, c.angle_q));
                const float norm = __fadd_rn(__fmul_rn(ni, ni), __fmul_rn(nq, nq));
                const float scalor = __fsub_rn(1.9999f, norm);
                cur_i = __fmul_rn(ni, scalor);
                cur_q = __fmul_rn(nq, scalor);
            }
            const float mi = __fsub_rn(__fmul_rn(v.x, my_i), __fmul_rn(v.y, my_q));
            const float mq = __fadd_rn(__fmul_rn(v.y, my_i), __fmul_rn(v.x, my_q));
            v = make_float2(mi, mq);
        }
        v.x = __double2float_rn(__dmul_rn((double)v.x, c.gain));
        v.y = __double2float_rn(__dmul_rn((double)v.y, c.gain));
        if (valid) row[k] = v;
    }
    if (lane == 0) {
        st->cur_i = cur_i;
        st->cur_q = cur_q;
        st->top_block = (top0 ^ n) & 1;
        st->fs4 = (fs40 + n) & 3;
    }
    if (row2)
        for (int i = lane; i < H; i += 32) st->hist[i] = ent[i];
}

// ---------------------------------------------------------------------------------------------------------------
// One-bin channels with a frequency offset (the usual case: a requested channel frequency is rarely the centre of its
// polyphase bin).  The oscillator is a float recursion -- rotate by the angle, fastNormalize -- that is neutrally stable
// in phase: two runs never merge, so unlike the Airspy DC filter it cannot be cut into speculative segments, and one
// chain step costs 44 cycles (12 fma-pipe instructions): 1.1 ms per 50 000-sample row, 14 x the whole polyphase
// kernel.  But the values do not depend on the samples.  osc_produce_kernel therefore runs AHEAD: after every call it
// tops a per-channel ring up to one call's worth of oscillator values on a side stream, one thread per channel, while
// the caller's FIR / demodulator kernels run; the call itself only does the element-wise osc_mix_kernel.
// (AbstractOscillator.mixComplex, J/dsp/mixer/AbstractOscillator.java:102-116: sample * current, then rotate();
// Oscillator.rotate + Complex.fastNormalize, J/dsp/mixer/Oscillator.java:42-68.)
// ---------------------------------------------------------------------------------------------------------------
struct MixChannel {
    int row;
    float angle_i, angle_q;
    double gain;
};

__global__ void __launch_bounds__(32) osc_produce_kernel(const MixChannel *__restrict__ chans, float2 *__restrict__ state,
                                                           float2 *__restrict__ ring, int ring_len, long long start, int count,
                                                           int n_mix)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_mix) return;
    const float angle_i = chans[ch].angle_i, angle_q = chans[ch].angle_q;
    float cur_i = state[ch].x, cur_q = state[ch].y;
    float2 *r = ring + (size_t)ch * ring_len;
    int pos = (int)(start % ring_len);
#define SDRGPU_OSC_ROTATE()                                                                        \
    {                                                                                              \
        const float ni = __fsub_rn(__fmul_rn(cur_i, angle_i), __fmul_rn(cur_q, angle_q));          \
        const float nq = __fadd_rn(__fmul_rn(cur_q, angle_i), __fmul_rn(cur_i, angle_q));          \
        const float scalor = __fsub_rn(1.9999f, __fadd_rn(__fmul_rn(ni, ni), __fmul_rn(nq, nq)));  \
        cur_i = __fmul_rn(ni, scalor);                                                             \
        cur_q = __fmul_rn(nq, scalor);                                                             \
    }
    int k = 0;
    while (k < count) {
        if ((pos & 1) == 0 && k + 8 <= count && pos + 8 <= ring_len) {
            // eight steps with nothing but the recursion between them, then four 16-byte stores (ring_len is even and
            // the rows are 16-byte aligned)
            float4 w[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                w[j].x = cur_i;
                w[j].y = cur_q;
                SDRGPU_OSC_ROTATE()
                w[j].z = cur_i;
                w[j].w = cur_q;
                SDRGPU_OSC_ROTATE()
            }
#pragma unroll
            for (int j = 0; j < 4; j++) reinterpret_cast<float4 *>(r + pos)[j] = w[j];
            pos += 8;
            k += 8;
        } else {
            r[pos] = make_float2(cur_i, cur_q);
            SDRGPU_OSC_ROTATE()
            pos += 1;
            k += 1;
        }
        if (pos >= ring_len) pos = 0;
    }
#undef SDRGPU_OSC_ROTATE
    state[ch] = make_float2(cur_i, cur_q);
}

// grid (ceil(n / 256), n_mix): row[k] = (float)((double)(row[k] * osc[start + k]) * gain)
__global__ void osc_mix_kernel(float *out, long long out_stride, const MixChannel *__restrict__ chans,
                               const float2 *__restrict__ ring, int ring_len, long long start, int n)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const MixChannel c = chans[blockIdx.y];
    float2 *row = reinterpret_cast<float2 *>(out + (size_t)c.row * out_stride);
    const float2 v = row[k];
    const float2 z = ring[(size_t)blockIdx.y * ring_len + (int)((start + k) % ring_len)];
    const float mi = __fsub_rn(__fmul_rn(v.x, z.x), __fmul_rn(v.y, z.y));
    const float mq = __fadd_rn(__fmul_rn(v.y, z.x), __fmul_rn(v.x, z.y));
    row[k] = make_float2(__double2float_rn(__dmul_rn((double)mi, c.gain)), __double2float_rn(__dmul_rn((double)mq, c.gain)));
}

// ---------------------------------------------------------------------------------------------------------------
// tuner sample converters (ByteSampleConverter / SignedByteSampleConverter lookup tables, ConversionUtils 16-bit)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float convert_value(int format, const void *src, size_t i)
{
    if (format == SDRGPU_FORMAT_U8) return __fdiv_rn((float)((int)reinterpret_cast<const uint8_t *>(src)[i] - 127), 128.0f);
    if (format == SDRGPU_FORMAT_S8) return __fdiv_rn((float)reinterpret_cast<const int8_t *>(src)[i], 128.0f);
    const uint8_t *b = reinterpret_cast<const uint8_t *>(src) + 2 * i;   // little endian, any alignment
    const short v = (short)((unsigned)b[0] | ((unsigned)b[1] << 8));
    return __fdiv_rn((float)v, 32767.0f);
}

__global__ void convert_kernel(int format, const void *__restrict__ src, float *__restrict__ dst, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = convert_value(format, src, i);
}

// new_state[i] = S[consumed + i], S = [state | in]
__global__ void save_state_kernel(const float2 *state, int state_len, const float2 *in, int n_in, int consumed,
                                  float2 *new_state, int new_len)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < new_len; i += gridDim.x * blockDim.x) {
        int idx = consumed + i;
        float2 v = make_float2(0.0f, 0.0f);
        if (idx < state_len) v = state[idx];
        else if (idx - state_len < n_in) v = in[idx - state_len];
        new_state[i] = v;
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------- handle
struct sdrgpu_channelizer {
    int device = 0;
    int M = 0, T = 0, half = 0, H = 0, NB = 16;
    int max_in_complex = 0, max_blocks = 0;
    int leftover = 0, parity0 = 0;
    bool throttled = false;   // chan_set_throttled: the pipeline is overlapping this launch with the demodulator
    // chan_convert leaves 8-bit tuner samples unconverted for chan_enqueue: the M = 400 / 800 filter bank converts them on
    // load (no float copy of the input in HBM); anything else converts them with convert_kernel first
    const uint8_t *defer_src = nullptr;
    const float2 *defer_dst = nullptr;
    int defer_n = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;   // H2D / D2H streams of the chunked host path
    cudaEvent_t events[kMaxEvents] = {};
    sdrgpu_status ensure_copy_streams()
    {
        if (copy_in) return SDRGPU_OK;
        SDRGPU_CUDA(cudaStreamCreateWithFlags(&copy_in, cudaStreamNonBlocking));
        SDRGPU_CUDA(cudaStreamCreateWithFlags(&copy_out, cudaStreamNonBlocking));
        for (auto &e : events) SDRGPU_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        return SDRGPU_OK;
    }
    float *d_taps = nullptr;
    float2 *d_tw = nullptr;
    float2 *d_tw2 = nullptr;   // pfb2_kernel inter-step twiddles
    int fast_r1 = 0, fast_r2 = 0;  // factors of the pfb2 fast path (0 = generic kernel)
    float2 *d_state[2] = {nullptr, nullptr};
    int cur_state = 0;
    float2 *d_in = nullptr;    // staging for host input (float I/Q)
    uint8_t *d_raw = nullptr;  // staging for host input in a native tuner format
    float2 *d_in_alt = nullptr;    // the other staging pair of an asynchronous pipeline (chan_swap_staging): the H2D copies of
    uint8_t *d_raw_alt = nullptr;  // call k + 1 land while the kernels of call k still read theirs
    int in_format = SDRGPU_FORMAT_F32;
    sdrgpu_airspy *airspy = nullptr;   // SDRGPU_FORMAT_AIRSPY_*: the stateful raw-sample converter
    float *d_out = nullptr;    // staging for host output
    size_t d_out_bytes = 0;
    int n_sel = 0;
    // every bin selected in order as a frequency-corrected one-bin channel with one float-representable gain (the usual
    // sdrtrunk situation when all channels of a tuner are in use): pfb2_kernel mixes the oscillators in where it stores
    int mix_identity = 0;
    float mix_gain = 0.0f;
    int *d_sel = nullptr;
    float *d_gain_f = nullptr;
    double *d_gain_d = nullptr;
    double sample_rate = 0.0;          // tuner sample rate (Hz); needed for frequency-corrected channels
    int n_rows = 0;                    // rows the pfb kernel writes: n_sel output rows + scratch rows of second bins
    int n_post = 0;                    // special channels (two-bin and / or frequency offset)
    PostChannel *d_post = nullptr;
    PostState *d_post_state = nullptr;
    float *d_out2 = nullptr;           // scratch rows [n_rows - n_sel][2 * max_blocks]
    // one-bin frequency-corrected channels: oscillator values produced ahead of use (osc_produce_kernel)
    int n_mix = 0, osc_ring_len = 0;
    MixChannel *d_mix = nullptr;
    float2 *d_mix_state = nullptr;     // oscillator vector at the producer's position
    float2 *d_osc = nullptr;           // [n_mix][osc_ring_len]
    long long osc_produced = 0, osc_consumed = 0, osc_safe = 0;   // osc_safe: produced by launches already waited for
    cudaStream_t osc_stream = nullptr;
    cudaEvent_t ev_mix = nullptr, ev_osc = nullptr;
    bool osc_pending = false;
    bool mix_recorded = false;   // ev_mix marks the end of the last kernel that read the rings
    SynthFilter synth{};
    int gain_exact = 1;
    int identity = 0;
    float gain_uniform = 0.0f;
    std::vector<sdrgpu_output_channel> channels;
    std::vector<int> factors;
    std::vector<unsigned> magic;
    size_t smem_bytes = 0;
    KernelTimer timer;
};

namespace {

sdrgpu_status upload_selection(sdrgpu_channelizer *h)
{
    const int n = (int)h->channels.size();
    std::vector<int> sel;
    std::vector<float> gf;
    std::vector<double> gd;
    std::vector<PostChannel> post;
    std::vector<MixChannel> mix;
    int exact = 1, n_two = 0;
    for (int i = 0; i < n; i++) {
        const sdrgpu_output_channel &c = h->channels[i];
        const bool special = c.bin2 >= 0 || c.frequency_offset_hz != 0;
        sel.push_back(c.bin1);
        // special rows leave the pfb kernel at gain 1; post_channel_kernel applies the gain after mixing
        gd.push_back(special ? 1.0 : c.gain);
        gf.push_back((float)gd.back());
        if ((double)gf.back() != gd.back()) exact = 0;
        if (special) {
            PostChannel pc{};
            pc.row = i;
            pc.row2 = c.bin2 >= 0 ? n_two++ : -1;
            // TwoChannelOutputProcessor mixes unconditionally, OneChannelOutputProcessor only with an offset
            pc.mix = 1;
            // Oscillator.update: anglePerSample = (float)(2 pi f / fs); Complex.fromAngle(float) -> (float)cos, (float)sin
            const double channel_rate = 2.0 * h->sample_rate / (double)h->M;
            const float angle = (float)(2.0 * 3.14159265358979323846 * (double)c.frequency_offset_hz / channel_rate);
            pc.angle_i = (float)cos((double)angle);
            pc.angle_q = (float)sin((double)angle);
            pc.gain = c.gain;
            if (c.bin2 >= 0) post.push_back(pc);                                        // two-bin: post_channel_kernel
            else mix.push_back(MixChannel{pc.row, pc.angle_i, pc.angle_q, pc.gain});    // one bin + offset: look-ahead
        }
    }
    for (int i = 0; i < n; i++)
        if (h->channels[i].bin2 >= 0) {   // scratch rows: the second bins, gain 1
            sel.push_back(h->channels[i].bin2);
            gd.push_back(1.0);
            gf.push_back(1.0f);
        }
    const int rows = (int)sel.size();
    h->mix_identity = (int)mix.size() == n && n == h->M && rows == n;
    for (size_t m = 0; m < mix.size() && h->mix_identity; m++)
        if (mix[m].row != (int)m || sel[m] != (int)m || mix[m].gain != mix[0].gain || (double)(float)mix[m].gain != mix[m].gain)
            h->mix_identity = 0;
    h->mix_gain = mix.empty() ? 0.0f : (float)mix[0].gain;
    cudaFree(h->d_sel);
    cudaFree(h->d_gain_f);
    cudaFree(h->d_gain_d);
    cudaFree(h->d_post);
    cudaFree(h->d_post_state);
    cudaFree(h->d_out2);
    if (h->osc_stream) SDRGPU_CUDA(cudaStreamSynchronize(h->osc_stream));
    cudaFree(h->d_mix);
    cudaFree(h->d_mix_state);
    cudaFree(h->d_osc);
    h->d_mix = nullptr;
    h->d_mix_state = nullptr;
    h->d_osc = nullptr;
    h->osc_produced = h->osc_consumed = h->osc_safe = 0;
    h->osc_pending = false;
    h->d_sel = nullptr;
    h->d_gain_f = nullptr;
    h->d_gain_d = nullptr;
    h->d_post = nullptr;
    h->d_post_state = nullptr;
    h->d_out2 = nullptr;
    SDRGPU_CUDA(cudaMalloc(&h->d_sel, sizeof(int) * (size_t)rows));
    SDRGPU_CUDA(cudaMalloc(&h->d_gain_f, sizeof(float) * (size_t)rows));
    SDRGPU_CUDA(cudaMalloc(&h->d_gain_d, sizeof(double) * (size_t)rows));
    SDRGPU_CUDA(cudaMemcpy(h->d_sel, sel.data(), sizeof(int) * (size_t)rows, cudaMemcpyHostToDevice));
    SDRGPU_CUDA(cudaMemcpy(h->d_gain_f, gf.data(), sizeof(float) * (size_t)rows, cudaMemcpyHostToDevice));
    SDRGPU_CUDA(cudaMemcpy(h->d_gain_d, gd.data(), sizeof(double) * (size_t)rows, cudaMemcpyHostToDevice));
    if (!post.empty()) {
        std::vector<PostState> init(post.size());
        std::memset(init.data(), 0, sizeof(PostState) * init.size());
        for (auto &st : init) {
            st.cur_i = 0.0f;   // Oscillator.java:24: mCurrentAngle = new Complex(0.0f, -1.0f)
            st.cur_q = -1.0f;
            st.top_block = 1;  // TwoChannelSynthesizerM2: mTopBlockIndicator = true
        }
        SDRGPU_CUDA(cudaMalloc(&h->d_post, sizeof(PostChannel) * post.size()));
        SDRGPU_CUDA(cudaMalloc(&h->d_post_state, sizeof(PostState) * post.size()));
        SDRGPU_CUDA(cudaMemcpy(h->d_post, post.data(), sizeof(PostChannel) * post.size(), cudaMemcpyHostToDevice));
        SDRGPU_CUDA(cudaMemcpy(h->d_post_state, init.data(), sizeof(PostState) * init.size(), cudaMemcpyHostToDevice));
    }
    if (n_two > 0) SDRGPU_CUDA(cudaMalloc(&h->d_out2, sizeof(float) * 2 * (size_t)h->max_blocks * (size_t)n_two));
    if (!mix.empty()) {
        if (!h->osc_stream) {
            SDRGPU_CUDA(cudaStreamCreateWithFlags(&h->osc_stream, cudaStreamNonBlocking));
            SDRGPU_CUDA(cudaEventCreateWithFlags(&h->ev_mix, cudaEventDisableTiming));
            SDRGPU_CUDA(cudaEventCreateWithFlags(&h->ev_osc, cudaEventDisableTiming));
        }
        // two calls' worth: a pipeline tops the ring up at the START of a call, for the call after it (chan_osc_ahead)
        h->osc_ring_len = (2 * h->max_blocks + 8 + 1) & ~1;   // even: the producer stores pairs
        std::vector<float2> start(mix.size(), make_float2(0.0f, -1.0f));   // Oscillator.java:24
        SDRGPU_CUDA(cudaMalloc(&h->d_mix, sizeof(MixChannel) * mix.size()));
        SDRGPU_CUDA(cudaMalloc(&h->d_mix_state, sizeof(float2) * mix.size()));
        SDRGPU_CUDA(cudaMalloc(&h->d_osc, sizeof(float2) * mix.size() * (size_t)h->osc_ring_len));
        SDRGPU_CUDA(cudaMemcpy(h->d_mix, mix.data(), sizeof(MixChannel) * mix.size(), cudaMemcpyHostToDevice));
        SDRGPU_CUDA(cudaMemcpy(h->d_mix_state, start.data(), sizeof(float2) * mix.size(), cudaMemcpyHostToDevice));
    }
    h->n_mix = (int)mix.size();
    h->n_sel = n;
    h->n_rows = rows;
    h->n_post = (int)post.size();
    h->gain_exact = exact;
    h->identity = exact && n == h->M && post.empty() && mix.empty();
    for (int i = 0; i < n && h->identity; i++)
        if (sel[i] != i || gf[i] != gf[0]) h->identity = 0;
    h->gain_uniform = n > 0 ? gf[0] : 0.0f;
    return SDRGPU_OK;
}

template <int M, int R1, int R2, int NB, int TT, int NT, int MINB, bool RAW = false>
sdrgpu_status launch_pfb2(const sdrgpu_channelizer *h, const ChanParams &p)
{
    using L = Pfb2Layout<M, R1, R2, NB, TT, NT>;
    auto kernel = pfb2_kernel<M, R1, R2, NB, TT, NT, MINB, RAW>;
    // a pipeline that overlaps its time chunks with the demodulator holds the channelizer to a few CTAs per SM
    // the direct row stores (NB = 8, default selection, channel layout) need no X region
    const size_t need = (p.identity && p.layout == SDRGPU_LAYOUT_CHANNELS) ? L::smem_direct : L::smem_bytes;
    const size_t smem = (h->throttled || g_tuning[SDRGPU_TUNE_THROTTLE_ALWAYS]) ? smem_for_ctas_per_sm(need, 0, g_tuning[SDRGPU_TUNE_PFB_CTAS_PER_SM]) : need;
    SDRGPU_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem > need ? 227 * 1024 : L::smem_bytes)));
    const int grid = (p.n_blocks + NB - 1) / NB;
    kernel<<<grid, NT, smem, h->stream>>>(p);
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    return SDRGPU_OK;
}

template <int NB, int TT>
sdrgpu_status launch_pfb(const sdrgpu_channelizer *h, const ChanParams &p, int grid)
{
    auto kernel = pfb_ifft_kernel<NB, TT>;
    SDRGPU_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes));
    kernel<<<grid, kThreads, h->smem_bytes, h->stream>>>(p);
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    return SDRGPU_OK;
}

}  // namespace

int sdrgpu::chan_selected_count(const sdrgpu_channelizer *h) { return h ? h->n_sel : 0; }

// Enqueues the channelizer kernels for n_in device-resident complex samples on the handle's stream and updates the
// host-side framing state (leftover samples, block parity, history ping-pong).  No copies, no synchronisation.
static void launch_convert(sdrgpu_channelizer *h, const uint8_t *src, float2 *dst, int n)
{
    const size_t values = 2 * (size_t)n;
    int grid = (int)((values + 255) / 256);
    if (grid > 148 * 16) grid = 148 * 16;
    convert_kernel<<<grid, 256, 0, h->stream>>>(h->in_format, src, reinterpret_cast<float *>(dst), values);
    count_launch();
}

sdrgpu_status sdrgpu::chan_enqueue(sdrgpu_channelizer *h, const float2 *d_in, int n_in, float *d_out, long long stride,
                                   int layout, int *n_blocks_out)
{
    const int total = h->leftover + n_in;
    const int n_blocks = total / h->half;
    if (n_blocks_out) *n_blocks_out = n_blocks;
    const float2 *state = h->d_state[h->cur_state];
    const int state_len = h->H + h->leftover;
    const int consumed = n_blocks * h->half;
    const int new_leftover = total - consumed;
    const int new_len = h->H + new_leftover;
    float2 *next = h->d_state[h->cur_state ^ 1];
    bool state_saved = false;
    // 8-bit samples chan_convert left unconverted: the filter bank reads them as they are when it runs, else convert now
    const uint8_t *raw = (h->defer_src && d_in == h->defer_dst && n_in == h->defer_n) ? h->defer_src : nullptr;
    h->defer_src = nullptr;
    const bool fuse_convert = raw && n_blocks > 0 && h->fast_r1 && (h->M == 400 || h->M == 800);
    if (raw && !fuse_convert) launch_convert(h, raw, const_cast<float2 *>(d_in), n_in);
    // checked before anything is launched or the framing state advances: a failing call leaves the handle as it was
    if (n_blocks > 0 && (h->n_mix > 0 || h->n_post > 0)) {
        // The reference rotates every channel's mixer for every buffer; the results layout has no per-channel rows to
        // mix, and skipping the oscillators would leave them out of step with the sample stream for later calls.
        if (layout != SDRGPU_LAYOUT_CHANNELS)
            return fail(SDRGPU_ERR_BAD_STATE, "two-bin / frequency-corrected channels are selected: use SDRGPU_LAYOUT_CHANNELS");
        if (h->n_mix > 0 && n_blocks > h->osc_ring_len)
            return fail(SDRGPU_ERR_OVERFLOW, "%d blocks exceed the oscillator look-ahead", n_blocks);
    }
    // Frequency-corrected one-bin channels: the oscillator values come from the look-ahead rings (osc_produce_kernel on a
    // side stream).  When every bin is such a channel pfb2_kernel multiplies them in where it stores the rows (no separate
    // pass over the channel streams); otherwise the rows leave the kernel at gain 1 and osc_mix_kernel finishes them.
    static const int fuse_mix_env = getenv("SDRGPU_FUSE_MIX") ? atoi(getenv("SDRGPU_FUSE_MIX")) : 1;
    // (pfb2_kernel instances with 8-block tiles store straight from step B: M = 160 ... 800, see the launch table below)
    const bool direct_store = h->fast_r1 && (h->M == 800 || h->M == 640 || h->M == 400 || h->M == 320 || h->M == 240 ||
                                             h->M == 200 || h->M == 160);
    const bool fused_mix = fuse_mix_env && h->n_mix > 0 && h->mix_identity && direct_store &&
                           layout == SDRGPU_LAYOUT_CHANNELS && n_blocks > 0;
    auto ensure_osc = [&]() -> sdrgpu_status {
        const int pgrid = (h->n_mix + 31) / 32;
        const long long have = h->osc_produced - h->osc_consumed;
        // wait for the top-up in flight only if this call reaches into what it writes (or has to produce itself)
        if (h->osc_pending && (h->osc_consumed + n_blocks > h->osc_safe || have < n_blocks)) {
            SDRGPU_CUDA(cudaStreamWaitEvent(h->stream, h->ev_osc, 0));
            h->osc_pending = false;
            h->osc_safe = h->osc_produced;
        }
        if (have < n_blocks) {  // first call, or a call longer than the look-ahead: produce the rest in line
            osc_produce_kernel<<<pgrid, 32, 0, h->stream>>>(h->d_mix, h->d_mix_state, h->d_osc, h->osc_ring_len,
                                                           h->osc_produced, (int)(n_blocks - have), h->n_mix);
            h->osc_produced += n_blocks - have;
            h->osc_safe = h->osc_produced;
            count_launch();
        }
        return SDRGPU_OK;
    };
    if (n_blocks > 0) {
        if (fused_mix) SDRGPU_TRY(ensure_osc());
        ChanParams p{};
        p.neg_zero = -0.0f;
        p.state = state;
        p.in = d_in;
        p.raw = fuse_convert ? raw : nullptr;
        p.raw_flip = h->in_format == SDRGPU_FORMAT_S8 ? 0x80 : 0;
        p.raw_bias = h->in_format == SDRGPU_FORMAT_S8 ? 128 : 127;
        p.taps = h->d_taps;
        p.tw = h->d_tw;
        p.tw2 = h->d_tw2;
        p.out = d_out;
        p.sel = h->d_sel;
        p.gain_f = h->d_gain_f;
        p.gain_d = h->d_gain_d;
        p.out_stride = stride;
        p.out2 = h->d_out2;
        p.out2_stride = 2LL * h->max_blocks;
        p.n_main = h->n_sel;
        p.state_len = state_len;
        p.n_in = n_in;
        p.M = h->M;
        p.T = h->T;
        p.half = h->half;
        p.H = h->H;
        p.n_blocks = n_blocks;
        p.parity0 = h->parity0;
        p.n_sel = h->n_rows;
        p.layout = layout;
        p.gain_exact = h->gain_exact;
        p.identity = fused_mix ? 1 : h->identity;   // (every bin in order, one gain: the direct store path, with the mix)
        p.osc = fused_mix ? h->d_osc : nullptr;
        p.osc_ring_len = h->osc_ring_len;
        p.osc_start = fused_mix ? (int)(h->osc_consumed % h->osc_ring_len) : 0;
        static const int pf_waves = getenv("SDRGPU_PFB_PREFETCH") ? atoi(getenv("SDRGPU_PFB_PREFETCH")) : 2;
        p.prefetch_blocks = 148 * 8 * pf_waves;   // in quarter waves of 148 SMs x 4 CTAs x 8 blocks
        p.gain_uniform = fused_mix ? h->mix_gain : h->gain_uniform;
        p.inv_m = 1.0f / (float)h->M;
        p.n_factors = (int)h->factors.size();
        for (int i = 0; i < p.n_factors; i++) {
            p.factors[i] = h->factors[i];
            p.magic_s[i] = h->magic[i];
        }
        const int grid = (n_blocks + h->NB - 1) / h->NB;
        if (h->fast_r1 && n_in > 0) {
            p.next_state = next;
            p.next_len = new_len;
            p.consumed = consumed;
            state_saved = true;
        }
        h->timer.begin(h->stream);
        sdrgpu_status st;
        // tile sizes measured on B200 (profiles/): M = 400 runs best as 8-block tiles, 200 threads, 4 CTAs per SM; M = 800 as
        // 8-block tiles, 256 threads, 3 CTAs per SM
        if (fuse_convert && h->M == 400) st = launch_pfb2<400, 20, 20, 8, 9, 200, 4, true>(h, p);
        else if (fuse_convert && h->M == 800) st = launch_pfb2<800, 32, 25, 8, 9, 256, 3, true>(h, p);
        else if (h->fast_r1 && h->M == 400) st = launch_pfb2<400, 20, 20, 8, 9, 200, 4>(h, p);
        else if (h->fast_r1 && h->M == 800) st = launch_pfb2<800, 32, 25, 8, 9, 256, 3>(h, p);
        else if (h->fast_r1 && h->M == 96) st = launch_pfb2<96, 8, 12, 16, 9, 192, 2>(h, p);
        else if (h->fast_r1 && h->M == 640) st = launch_pfb2<640, 32, 20, 8, 9, 320, 2>(h, p);
        else if (h->fast_r1 && h->M == 320) st = launch_pfb2<320, 16, 20, 8, 9, 160, 4>(h, p);
        else if (h->fast_r1 && h->M == 240) st = launch_pfb2<240, 12, 20, 8, 9, 160, 4>(h, p);
        else if (h->fast_r1 && h->M == 200) st = launch_pfb2<200, 10, 20, 8, 9, 160, 4>(h, p);
        else if (h->fast_r1 && h->M == 160) st = launch_pfb2<160, 8, 20, 8, 9, 160, 4>(h, p);
        else if (h->fast_r1 && h->M == 120) st = launch_pfb2<120, 10, 12, 16, 9, 192, 2>(h, p);
        else if (h->fast_r1 && h->M == 100) st = launch_pfb2<100, 10, 10, 16, 9, 160, 2>(h, p);
        else if (h->fast_r1 && h->M == 80) st = launch_pfb2<80, 8, 10, 16, 9, 160, 2>(h, p);
        else if (h->NB == 16) st = (h->T == 9) ? launch_pfb<16, 9>(h, p, grid) : launch_pfb<16, 0>(h, p, grid);
        else st = (h->T == 9) ? launch_pfb<8, 9>(h, p, grid) : launch_pfb<8, 0>(h, p, grid);
        h->timer.end(h->stream);
        SDRGPU_TRY(st);
        if (layout == SDRGPU_LAYOUT_CHANNELS && h->n_post > 0) {
            post_channel_kernel<<<h->n_post, 32, 0, h->stream>>>(d_out, stride, h->d_out2, 2LL * h->max_blocks, n_blocks, h->d_post,
                                                                 h->d_post_state, h->synth);
            count_launch();
            SDRGPU_CUDA(cudaGetLastError());
        }
        if (layout == SDRGPU_LAYOUT_CHANNELS && h->n_mix > 0) {
            if (!fused_mix) {
                SDRGPU_TRY(ensure_osc());
                osc_mix_kernel<<<dim3((n_blocks + 255) / 256, h->n_mix), 256, 0, h->stream>>>(d_out, stride, h->d_mix, h->d_osc,
                                                                                              h->osc_ring_len, h->osc_consumed, n_blocks);
                count_launch();
            }
            h->osc_consumed += n_blocks;
            SDRGPU_CUDA(cudaEventRecord(h->ev_mix, h->stream));
            h->mix_recorded = true;
            // top the ring up to a call's worth on the side stream, behind the kernel that has just read it
            const int pgrid = (h->n_mix + 31) / 32;
            const int top_up = h->max_blocks - (int)(h->osc_produced - h->osc_consumed);
            if (top_up > 0) {
                SDRGPU_CUDA(cudaStreamWaitEvent(h->osc_stream, h->ev_mix, 0));
                // Round 1 kept other blocks off the producer's SMs by asking for 220 KB of shared memory it never touched
                // (SDRGPU_OSC_EXCLUSIVE=1 still does); that only worked for one pipeline per GPU and starves everything else
                // once several tuners share the device, so the producer is an ordinary small kernel on its side stream and
                // the cost is reported as measured (bench.py: with_frequency_corrected_channels).
                static const int exclusive = getenv("SDRGPU_OSC_EXCLUSIVE") ? atoi(getenv("SDRGPU_OSC_EXCLUSIVE")) : 0;
                const int smem = (exclusive && pgrid <= 16) ? 220 * 1024 : 0;
                if (smem) SDRGPU_CUDA(cudaFuncSetAttribute(osc_produce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
                osc_produce_kernel<<<pgrid, 32, smem, h->osc_stream>>>(h->d_mix, h->d_mix_state, h->d_osc, h->osc_ring_len,
                                                                       h->osc_produced, top_up, h->n_mix);
                SDRGPU_CUDA(cudaEventRecord(h->ev_osc, h->osc_stream));
                h->osc_produced += top_up;
                h->osc_pending = true;
                count_launch();
            }
            SDRGPU_CUDA(cudaGetLastError());
        }
    }
    // carry the history + leftover over to the next call
    if (n_in > 0) {
        if (!state_saved) {
            int grid = (new_len + 255) / 256;
            if (grid > 1024) grid = 1024;
            save_state_kernel<<<grid, 256, 0, h->stream>>>(state, state_len, d_in, n_in, consumed, next, new_len);
            count_launch();
            SDRGPU_CUDA(cudaGetLastError());
        }
        h->cur_state ^= 1;
    }
    h->leftover = new_leftover;
    h->parity0 = (h->parity0 + n_blocks) & 1;
    return SDRGPU_OK;
}

cudaStream_t sdrgpu::chan_stream(const sdrgpu_channelizer *h) { return h->stream; }

size_t sdrgpu::chan_complex_bytes(const sdrgpu_channelizer *h)
{
    switch (h->in_format) {
    case SDRGPU_FORMAT_F32: return 8;
    case SDRGPU_FORMAT_S16LE: return 4;
    case SDRGPU_FORMAT_AIRSPY_U16LE: return 4;       // two real samples of two bytes
    case SDRGPU_FORMAT_AIRSPY_PACKED12: return 3;    // two real samples in three bytes
    default: return 2;
    }
}

sdrgpu_status sdrgpu::chan_upload(sdrgpu_channelizer *h, const void *iq, size_t first, int n, cudaStream_t copy_stream)
{
    const size_t cb = chan_complex_bytes(h);
    if (!h->d_in) SDRGPU_CUDA(cudaMalloc(&h->d_in, sizeof(float2) * (size_t)h->max_in_complex));
    void *dst = h->d_in + first;
    if (h->in_format != SDRGPU_FORMAT_F32) {
        // sized for the widest native format, so that the format can change without reallocating
        if (!h->d_raw) SDRGPU_CUDA(cudaMalloc(&h->d_raw, 4 * (size_t)h->max_in_complex));
        dst = h->d_raw + cb * first;
    }
    SDRGPU_CUDA(cudaMemcpyAsync(dst, reinterpret_cast<const uint8_t *>(iq) + cb * first, cb * (size_t)n,
                                cudaMemcpyHostToDevice, copy_stream));
    return SDRGPU_OK;
}

const float2 *sdrgpu::chan_convert(sdrgpu_channelizer *h, const void *iq_device, size_t first, int n)
{
    const size_t cb = chan_complex_bytes(h);
    if (h->in_format == SDRGPU_FORMAT_F32)
        return iq_device ? reinterpret_cast<const float2 *>(iq_device) + first : h->d_in + first;
    if (!h->d_in && cudaMalloc(&h->d_in, sizeof(float2) * (size_t)h->max_in_complex) != cudaSuccess) return nullptr;
    const uint8_t *src = iq_device ? reinterpret_cast<const uint8_t *>(iq_device) : h->d_raw;
    if (n > 0 && h->airspy) {
        // two real samples per complex sample: unpack, DC removal, Hilbert transform (airspy.cu), in stream order
        if (airspy_enqueue(h->airspy, src + cb * first, 2 * n, h->in_format == SDRGPU_FORMAT_AIRSPY_PACKED12, h->d_in + first,
                           h->stream) != SDRGPU_OK)
            return nullptr;
    } else if (n > 0) {
        const bool eight_bit = h->in_format == SDRGPU_FORMAT_U8 || h->in_format == SDRGPU_FORMAT_S8;
        static const int fuse_env = getenv("SDRGPU_FUSE_CONVERT") ? atoi(getenv("SDRGPU_FUSE_CONVERT")) : 1;
        if (fuse_env && eight_bit && h->fast_r1 && (h->M == 400 || h->M == 800)) {
            h->defer_src = src + cb * first;
            h->defer_dst = h->d_in + first;
            h->defer_n = n;
        } else {
            launch_convert(h, src + cb * first, h->d_in + first, n);
        }
    }
    return h->d_in + first;
}
// Oscillator look-ahead of a pipeline: at the START of a call (before its channelizer kernels) the rings are topped up to
// two calls' worth, i.e. the values of the NEXT call are produced beside this call's channelizer / first FIR launches --
// throughput-bound kernels that lose little to 200 latency-bound warps -- instead of behind them, beside the demodulator,
// whose launch time is set by its most loaded scheduler (8 tuners, all 6400 channels corrected: 9.1 -> see DESIGN.md).
sdrgpu_status sdrgpu::chan_osc_ahead(sdrgpu_channelizer *h)
{
    static const int ahead_env = getenv("SDRGPU_OSC_AHEAD") ? atoi(getenv("SDRGPU_OSC_AHEAD")) : 1;
    if (!ahead_env || h->n_mix <= 0 || !h->d_osc) return SDRGPU_OK;
    const int top_up = 2 * h->max_blocks - (int)(h->osc_produced - h->osc_consumed);
    if (top_up <= 0) return SDRGPU_OK;
    // the producer in flight (this call's values) first: ev_osc is about to be re-recorded
    if (h->osc_pending) {
        SDRGPU_CUDA(cudaStreamWaitEvent(h->stream, h->ev_osc, 0));
        h->osc_pending = false;
        h->osc_safe = h->osc_produced;
    }
    if (h->mix_recorded) SDRGPU_CUDA(cudaStreamWaitEvent(h->osc_stream, h->ev_mix, 0));   // the slots' last reader
    osc_produce_kernel<<<(h->n_mix + 31) / 32, 32, 0, h->osc_stream>>>(h->d_mix, h->d_mix_state, h->d_osc, h->osc_ring_len,
                                                                       h->osc_produced, top_up, h->n_mix);
    SDRGPU_CUDA(cudaGetLastError());
    SDRGPU_CUDA(cudaEventRecord(h->ev_osc, h->osc_stream));
    h->osc_produced += top_up;
    h->osc_pending = true;
    count_launch();
    return SDRGPU_OK;
}

cudaStream_t sdrgpu::chan_osc_stream(const sdrgpu_channelizer *h) { return h->n_mix > 0 ? h->osc_stream : nullptr; }

void sdrgpu::chan_swap_staging(sdrgpu_channelizer *h)
{
    std::swap(h->d_in, h->d_in_alt);
    std::swap(h->d_raw, h->d_raw_alt);
}
// where chan_upload puts a host buffer: device-resident input in the handle's sample format
const void *sdrgpu::chan_staging(const sdrgpu_channelizer *h)
{
    return h->in_format == SDRGPU_FORMAT_F32 ? static_cast<const void *>(h->d_in) : static_cast<const void *>(h->d_raw);
}
void sdrgpu::chan_set_throttled(sdrgpu_channelizer *h, bool on) { h->throttled = on; }
int sdrgpu::chan_half(const sdrgpu_channelizer *h) { return h->half; }
int sdrgpu::chan_max_in(const sdrgpu_channelizer *h) { return h->max_in_complex; }
int sdrgpu::chan_leftover(const sdrgpu_channelizer *h) { return h->leftover; }


extern "C" {

sdrgpu_status sdrgpu_chan_create(sdrgpu_channelizer **out, const float *taps, int n_taps, int channel_count,
                                 int max_input_floats)
{
    if (!out || !taps || n_taps <= 0) return fail(SDRGPU_ERR_INVALID_ARG, "NULL / empty argument");
    if (channel_count <= 0 || channel_count % 2 != 0)
        return fail(SDRGPU_ERR_INVALID_ARG, "Channel count must be an even multiple of the over-sample rate (2x)");
    if (max_input_floats <= 0 || max_input_floats % 2 != 0)
        return fail(SDRGPU_ERR_INVALID_ARG, "max_input_floats must be a positive even number");
    int dev = 0;
    SDRGPU_CUDA(cudaGetDevice(&dev));
    auto *h = new sdrgpu_channelizer();
    h->device = dev;
    const int M = channel_count;
    h->M = M;
    h->half = M / 2;
    // ComplexPolyphaseChannelizerM2.java:102: mTapsPerChannel = ceil(taps.length / channelCount)
    h->T = (n_taps + M - 1) / M;
    h->H = (2 * h->T - 1) * h->half;
    h->max_in_complex = max_input_floats / 2;
    h->max_blocks = (h->max_in_complex + h->half) / h->half;

    // FFT plan: radix 4, 2, 3, 5 then remaining odd primes (same factor preference as FFTPACK / JTransforms)
    int rem = M;
    const int pref[4] = {4, 2, 3, 5};
    for (int f : pref)
        while (rem % f == 0) {
            h->factors.push_back(f);
            rem /= f;
        }
    for (int f = 7; rem > 1; f += 2)
        while (rem % f == 0) {
            h->factors.push_back(f);
            rem /= f;
        }
    if ((int)h->factors.size() > kMaxFactors) {
        delete h;
        return fail(SDRGPU_ERR_INVALID_ARG, "channel count %d has too many prime factors", M);
    }
    int s = 1;
    for (int f : h->factors) {
        h->magic.push_back((unsigned)((0x100000000ULL + (unsigned long long)s - 1) / (unsigned long long)s));
        s *= f;
    }

    // tile of NB blocks per CTA: 16 when two ping-pong buffers of [M][NB+1] float2 fit in ~110 KB, else 8
    auto smem_for = [&](int nb) { return (size_t)(2 * (size_t)M * (nb + 1) + (size_t)M) * sizeof(float2); };
    h->NB = 16;
    if (smem_for(16) > 112 * 1024) h->NB = 8;
    h->smem_bytes = smem_for(h->NB);
    if (h->smem_bytes > 227 * 1024) {
        delete h;
        return fail(SDRGPU_ERR_INVALID_ARG, "channel count %d too large for the shared-memory FFT", M);
    }

    std::vector<float> padded((size_t)M * h->T, 0.0f);
    for (int i = 0; i < n_taps; i++) padded[i] = taps[i];
    std::vector<float2> tw(M);
    for (int k = 0; k < M; k++) {
        double a = 2.0 * 3.14159265358979323846 * (double)k / (double)M;
        tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    sdrgpu_status st = SDRGPU_OK;
    auto cleanup_fail = [&](sdrgpu_status code) {
        sdrgpu_chan_destroy(h);
        return code;
    };
#define CHK(call)                                                                                             \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess)                                                                               \
            return cleanup_fail(fail(SDRGPU_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__)));      \
    } while (0)
    CHK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    CHK(cudaMalloc(&h->d_taps, sizeof(float) * padded.size()));
    CHK(cudaMemcpy(h->d_taps, padded.data(), sizeof(float) * padded.size(), cudaMemcpyHostToDevice));
    CHK(cudaMalloc(&h->d_tw, sizeof(float2) * (size_t)M));
    CHK(cudaMemcpy(h->d_tw, tw.data(), sizeof(float2) * (size_t)M, cudaMemcpyHostToDevice));
    // fast path (pfb2_kernel) for the channel counts of the common tuner rates with the reference's 9 taps per channel
    if (h->T == 9) {
        // channel counts of the common tuner rates (25 kHz channels): 2 / 2.4 / 2.5 / 3 / 4 / 5 / 6 / 8 / 10 / 16 / 20 MS/s
        static const int fast[][3] = {{400, 20, 20}, {800, 32, 25}, {96, 8, 12}, {640, 32, 20}, {320, 16, 20}, {240, 12, 20}, {200, 10, 20}, {160, 8, 20}, {120, 10, 12}, {100, 10, 10}, {80, 8, 10}};
        for (const auto &f : fast)
            if (M == f[0]) {
                h->fast_r1 = f[1];
                h->fast_r2 = f[2];
            }
    }
    if (h->fast_r1) {
        std::vector<float2> tw2((size_t)M);
        for (int k1 = 0; k1 < h->fast_r1; k1++)
            for (int n2 = 0; n2 < h->fast_r2; n2++) {
                const double a = 2.0 * 3.14159265358979323846 * (double)((long long)k1 * n2 % M) / (double)M;
                tw2[(size_t)k1 * h->fast_r2 + n2] = make_float2((float)cos(a), (float)sin(a));
            }
        CHK(cudaMalloc(&h->d_tw2, sizeof(float2) * (size_t)M));
        CHK(cudaMemcpy(h->d_tw2, tw2.data(), sizeof(float2) * (size_t)M, cudaMemcpyHostToDevice));
    }
    const size_t state_cap = (size_t)h->H + h->half;
    for (int i = 0; i < 2; i++) {
        CHK(cudaMalloc(&h->d_state[i], sizeof(float2) * state_cap));
        CHK(cudaMemset(h->d_state[i], 0, sizeof(float2) * state_cap));
    }
#undef CHK
    h->channels.resize(M);
    for (int k = 0; k < M; k++) h->channels[k] = sdrgpu_output_channel{k, -1, 0, (double)M};
    st = upload_selection(h);
    if (st != SDRGPU_OK) return cleanup_fail(st);
    *out = h;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_chan_destroy(sdrgpu_channelizer *h)
{
    if (!h) return SDRGPU_OK;
    // a caller-owned stream may already be gone: never touch it here, wait for the device instead
    if (h->stream && h->stream != h->own_stream) cudaDeviceSynchronize();
    else if (h->own_stream) cudaStreamSynchronize(h->own_stream);
    cudaFree(h->d_taps);
    cudaFree(h->d_tw);
    cudaFree(h->d_tw2);
    cudaFree(h->d_state[0]);
    cudaFree(h->d_state[1]);
    cudaFree(h->d_in);
    cudaFree(h->d_raw);
    cudaFree(h->d_in_alt);
    cudaFree(h->d_raw_alt);
    sdrgpu::airspy_destroy(h->airspy);
    cudaFree(h->d_out);
    cudaFree(h->d_sel);
    cudaFree(h->d_gain_f);
    cudaFree(h->d_gain_d);
    cudaFree(h->d_post);
    cudaFree(h->d_post_state);
    cudaFree(h->d_out2);
    if (h->osc_stream) {
        cudaStreamSynchronize(h->osc_stream);
        cudaStreamDestroy(h->osc_stream);
        cudaEventDestroy(h->ev_mix);
        cudaEventDestroy(h->ev_osc);
    }
    cudaFree(h->d_mix);
    cudaFree(h->d_mix_state);
    cudaFree(h->d_osc);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->copy_in) cudaStreamDestroy(h->copy_in);
    if (h->copy_out) cudaStreamDestroy(h->copy_out);
    for (auto &e : h->events)
        if (e) cudaEventDestroy(e);
    delete h;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_chan_set_stream(sdrgpu_channelizer *h, void *cuda_stream)
{
    if (!h) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    cudaStream_t next = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    if (next == h->stream) return SDRGPU_OK;
    SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
    h->stream = next;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_chan_sync(sdrgpu_channelizer *h)
{
    if (!h) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_chan_set_input_format(sdrgpu_channelizer *h, int format)
{
    if (!h) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    if (format < SDRGPU_FORMAT_F32 || format > SDRGPU_FORMAT_AIRSPY_PACKED12)
        return fail(SDRGPU_ERR_INVALID_ARG, "unknown sample format %d", format);
    SDRGPU_CUDA(cudaSetDevice(h->device));
    SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
    const bool airspy = format == SDRGPU_FORMAT_AIRSPY_U16LE || format == SDRGPU_FORMAT_AIRSPY_PACKED12;
    const bool was = h->in_format == SDRGPU_FORMAT_AIRSPY_U16LE || h->in_format == SDRGPU_FORMAT_AIRSPY_PACKED12;
    if (airspy && !h->airspy) SDRGPU_TRY(sdrgpu::airspy_create(&h->airspy, 2 * h->max_in_complex));
    if (!airspy && h->airspy) {   // a later return to the Airspy formats starts from a fresh converter
        sdrgpu::airspy_destroy(h->airspy);
        h->airspy = nullptr;
    }
    (void)was;   // switching between the two Airspy packings keeps the converter state (setSamplePacking)
    h->in_format = format;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_convert_samples(int format, const void *src, int src_mem, int n_values, float *dst, int dst_mem)
{
    if (format < SDRGPU_FORMAT_U8 || format > SDRGPU_FORMAT_S16LE) return fail(SDRGPU_ERR_INVALID_ARG, "unknown native sample format %d", format);
    if (n_values < 0 || (n_values > 0 && (!src || !dst))) return fail(SDRGPU_ERR_INVALID_ARG, "NULL / negative argument");
    if (n_values == 0) return SDRGPU_OK;
    const size_t vb = format == SDRGPU_FORMAT_S16LE ? 2 : 1;
    // device staging for host buffers: kept per host thread and grown on demand (a converter is called once per tuner
    // buffer; an allocation per call would cost more than the conversion)
    struct Staging {
        void *p = nullptr;
        size_t cap = 0;
        int device = -1;
        cudaError_t ensure(size_t bytes)
        {
            int dev = 0;
            cudaGetDevice(&dev);
            if (p && (dev != device || bytes > cap)) {
                cudaFree(p);
                p = nullptr;
            }
            if (p) return cudaSuccess;
            device = dev;
            cap = bytes;
            return cudaMalloc(&p, bytes);
        }
    };
    static thread_local Staging stage_src, stage_dst;
    void *d_src = const_cast<void *>(src);
    float *d_dst = dst;
    if (src_mem == SDRGPU_HOST) {
        SDRGPU_CUDA(stage_src.ensure(vb * (size_t)n_values));
        d_src = stage_src.p;
        SDRGPU_CUDA(cudaMemcpy(d_src, src, vb * (size_t)n_values, cudaMemcpyHostToDevice));
    }
    if (dst_mem == SDRGPU_HOST) {
        SDRGPU_CUDA(stage_dst.ensure(sizeof(float) * (size_t)n_values));
        d_dst = static_cast<float *>(stage_dst.p);
    }
    int grid = (n_values + 255) / 256;
    if (grid > 148 * 16) grid = 148 * 16;
    convert_kernel<<<grid, 256>>>(format, d_src, d_dst, (size_t)n_values);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && dst_mem == SDRGPU_HOST) e = cudaMemcpy(dst, d_dst, sizeof(float) * (size_t)n_values, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(SDRGPU_ERR_CUDA, "sample conversion failed: %s", cudaGetErrorString(e));
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_chan_set_sample_rate(sdrgpu_channelizer *h, double sample_rate)
{
    if (!h) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    if (!(sample_rate > 0.0)) return fail(SDRGPU_ERR_INVALID_ARG, "sample rate must be positive");
    const bool changed = sample_rate != h->sample_rate;
    h->sample_rate = sample_rate;
    // the oscillator angles of frequency-corrected / two-bin channels depend on the channel rate: re-derive them
    // (like Oscillator.setSampleRate -> update(); this restarts the oscillators, as selecting does)
    if (changed && (h->n_mix > 0 || h->n_post > 0)) {
        SDRGPU_CUDA(cudaSetDevice(h->device));
        SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
        return upload_selection(h);
    }
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_chan_select(sdrgpu_channelizer *h, const sdrgpu_output_channel *channels, int n_channels,
                                 const float *synthesis_filter, int n_synthesis_taps)
{
    if (!h || !channels || n_channels <= 0) return fail(SDRGPU_ERR_INVALID_ARG, "NULL / empty selection");
    bool any_two = false, any_special = false;
    for (int i = 0; i < n_channels; i++) {
        if (channels[i].bin1 < 0 || channels[i].bin1 >= h->M)
            return fail(SDRGPU_ERR_INVALID_ARG, "Channel [%d] is not valid -- max channel is %d", channels[i].bin1, h->M);
        if (channels[i].bin2 >= h->M)
            return fail(SDRGPU_ERR_INVALID_ARG, "Channel [%d] is not valid -- max channel is %d", channels[i].bin2, h->M);
        any_two |= channels[i].bin2 >= 0;
        any_special |= channels[i].bin2 >= 0 || channels[i].frequency_offset_hz != 0;
    }
    if (any_special && !(h->sample_rate > 0.0))
        return fail(SDRGPU_ERR_BAD_STATE, "two-bin / frequency-corrected channels need sdrgpu_chan_set_sample_rate first");
    if (any_two) {
        if (!synthesis_filter || n_synthesis_taps < 2)
            return fail(SDRGPU_ERR_INVALID_ARG, "two-bin channels need the synthesis filter (getSincM2Synthesizer)");
        // TwoChannelSynthesizerM2.init (:74-88): tapsPerChannel = ceil(filter.length / 2) with integer division; the
        // I/Q-duplicated filter has 2 * tapsPerChannel * 2 entries
        const int entries = n_synthesis_taps / 2;
        if (entries > kMaxSynthEntries)
            return fail(SDRGPU_ERR_INVALID_ARG, "synthesis filter longer than %d taps", 2 * kMaxSynthEntries);
        std::memset(&h->synth, 0, sizeof(h->synth));
        h->synth.entries = entries;
        int fp = 0;
        for (int cp = 0; cp < n_synthesis_taps && fp + 1 < 4 * entries; cp++) {
            h->synth.f[fp++] = synthesis_filter[cp];
            h->synth.f[fp++] = synthesis_filter[cp];
        }
    }
    SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
    h->channels.assign(channels, channels + n_channels);
    return upload_selection(h);
}

int sdrgpu_chan_blocks_for(const sdrgpu_channelizer *h, int n_floats)
{
    if (!h || n_floats < 0) return 0;
    return (h->leftover + n_floats / 2) / h->half;
}

sdrgpu_status sdrgpu_chan_enable_timing(sdrgpu_channelizer *h, int enable)
{
    if (!h) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    return h->timer.enable(enable != 0);
}

sdrgpu_status sdrgpu_chan_last_kernel_ms(sdrgpu_channelizer *h, float *ms)
{
    if (!h || !ms) return fail(SDRGPU_ERR_INVALID_ARG, "NULL argument");
    return h->timer.read(ms);
}

sdrgpu_status sdrgpu_chan_process(sdrgpu_channelizer *h, const void *iq, int n_floats, int in_mem, float *out,
                                  long long out_stride_floats, int out_mem, int layout, int *n_blocks_out)
{
    if (!h) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    if (n_floats < 0 || n_floats % 2 != 0) return fail(SDRGPU_ERR_INVALID_ARG, "n_floats must be even (interleaved I/Q)");
    if (n_floats > 0 && !iq) return fail(SDRGPU_ERR_INVALID_ARG, "iq is NULL");
    if (layout != SDRGPU_LAYOUT_RESULTS && layout != SDRGPU_LAYOUT_CHANNELS)
        return fail(SDRGPU_ERR_INVALID_ARG, "unknown layout %d", layout);
    const int n_in = n_floats / 2;
    if (n_in > h->max_in_complex)
        return fail(SDRGPU_ERR_OVERFLOW, "input of %d floats exceeds the handle's max_input_floats %d", n_floats,
                    2 * h->max_in_complex);
    if (((uintptr_t)iq & 7) != 0 && in_mem == SDRGPU_DEVICE && h->in_format == SDRGPU_FORMAT_F32)
        return fail(SDRGPU_ERR_INVALID_ARG, "device input must be 8-byte aligned");
    SDRGPU_CUDA(cudaSetDevice(h->device));

    const int total = h->leftover + n_in;
    const int n_blocks = total / h->half;
    if (n_blocks_out) *n_blocks_out = n_blocks;
    const int rows = (layout == SDRGPU_LAYOUT_CHANNELS) ? h->n_sel : 0;
    if (n_blocks > 0) {
        if (!out) return fail(SDRGPU_ERR_INVALID_ARG, "out is NULL");
        if (layout == SDRGPU_LAYOUT_CHANNELS && (out_stride_floats < 2LL * n_blocks || (out_stride_floats & 1)))
            return fail(SDRGPU_ERR_INVALID_ARG, "out_stride_floats must be even and >= 2 * n_blocks (%d)", 2 * n_blocks);
        if (out_mem == SDRGPU_DEVICE && ((uintptr_t)out & 7) != 0)
            return fail(SDRGPU_ERR_INVALID_ARG, "device output must be 8-byte aligned");
    }

    // device staging for host buffers
    float *d_out = out;
    long long stride = out_stride_floats;
    if (out_mem == SDRGPU_HOST && n_blocks > 0) {
        const size_t need = (layout == SDRGPU_LAYOUT_CHANNELS) ? sizeof(float) * 2 * (size_t)n_blocks * (size_t)rows
                                                              : sizeof(float) * 2 * (size_t)n_blocks * (size_t)h->M;
        if (need > h->d_out_bytes) {
            if (h->d_out) {
                SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
                cudaFree(h->d_out);
                h->d_out = nullptr;
            }
            const size_t cap = sizeof(float) * 2 * (size_t)h->max_blocks * (size_t)(h->M > h->n_sel ? h->M : h->n_sel);
            const size_t bytes = need > cap ? need : cap;
            SDRGPU_CUDA(cudaMalloc(&h->d_out, bytes));
            h->d_out_bytes = bytes;
        }
        d_out = h->d_out;
        stride = 2LL * n_blocks;
    }
    if (in_mem == SDRGPU_DEVICE && out_mem == SDRGPU_DEVICE) {
        int got = 0;
        const float2 *src = sdrgpu::chan_convert(h, iq, 0, n_in);
        if (!src && n_in > 0) return fail(SDRGPU_ERR_NOMEM, "cannot allocate the input staging buffer");
        return sdrgpu::chan_enqueue(h, src, n_in, out, out_stride_floats, layout, &got);
    }

    // Host buffers: the call is cut into chunks so that the H2D copy of chunk i+1, the kernels of chunk i and the D2H
    // copy of chunk i-1 overlap on three streams (PCIe is full duplex; the copies, not the kernels, bound this path).
    // Block framing carries over between chunks exactly as between calls, so the result does not depend on the cut.
    SDRGPU_TRY(h->ensure_copy_streams());
    const int tile = h->half * 64;                                    // whole tiles of the kernels
    int chunk = (n_in + 7) / 8;
    chunk = (chunk + tile - 1) / tile * tile;
    if (chunk < tile) chunk = tile;
    // the first two chunks are a quarter of the rest: the D2H stream (the bottleneck) starts sooner
    int small = (chunk / 4 + tile - 1) / tile * tile;
    if (small < tile) small = tile;
    int done_in = 0, done_blocks = 0, ci = 0;
    while (done_in < n_in || (n_in == 0 && ci == 0)) {
        const int want = ci < 2 ? small : chunk;
        const int n = (n_in - done_in < want) ? n_in - done_in : want;
        const float2 *src_dev = nullptr;
        cudaEvent_t ev_in = h->events[(2 * ci) % kMaxEvents], ev_k = h->events[(2 * ci + 1) % kMaxEvents];
        if (in_mem == SDRGPU_HOST && n > 0) {
            SDRGPU_TRY(sdrgpu::chan_upload(h, iq, (size_t)done_in, n, h->copy_in));
            SDRGPU_CUDA(cudaEventRecord(ev_in, h->copy_in));
            SDRGPU_CUDA(cudaStreamWaitEvent(h->stream, ev_in, 0));
            src_dev = sdrgpu::chan_convert(h, nullptr, (size_t)done_in, n);
        } else {
            src_dev = sdrgpu::chan_convert(h, iq, (size_t)done_in, n);
        }
        if (!src_dev && n > 0) return fail(SDRGPU_ERR_NOMEM, "cannot allocate the input staging buffer");
        float *dst = nullptr;
        if (n_blocks > 0)
            dst = (layout == SDRGPU_LAYOUT_CHANNELS) ? d_out + 2 * (size_t)done_blocks : d_out + 2 * (size_t)done_blocks * h->M;
        int got = 0;
        SDRGPU_TRY(sdrgpu::chan_enqueue(h, src_dev, n, dst, stride, layout, &got));
        if (out_mem == SDRGPU_HOST && got > 0) {
            SDRGPU_CUDA(cudaEventRecord(ev_k, h->stream));
            SDRGPU_CUDA(cudaStreamWaitEvent(h->copy_out, ev_k, 0));
            if (layout == SDRGPU_LAYOUT_CHANNELS) {
                SDRGPU_CUDA(cudaMemcpy2DAsync(out + 2 * (size_t)done_blocks, sizeof(float) * (size_t)out_stride_floats, dst,
                                              sizeof(float) * (size_t)stride, sizeof(float) * 2 * (size_t)got, (size_t)rows,
                                              cudaMemcpyDeviceToHost, h->copy_out));
            } else {
                SDRGPU_CUDA(cudaMemcpyAsync(out + 2 * (size_t)done_blocks * h->M, dst, sizeof(float) * 2 * (size_t)got * (size_t)h->M,
                                            cudaMemcpyDeviceToHost, h->copy_out));
            }
        }
        done_in += n;
        done_blocks += got;
        ci++;
        if (n_in == 0) break;
    }
    SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
    if (out_mem == SDRGPU_HOST) SDRGPU_CUDA(cudaStreamSynchronize(h->copy_out));
    return SDRGPU_OK;
}

}  // extern "C"
