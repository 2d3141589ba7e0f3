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
#include <cstring>
#include <utility>
#include <vector>

#include "common.cuh"
#include "fft_regs.cuh"
#include "outputs.cuh"

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
    // the ROUTED kernel instances: row c < n_main goes to rows[c] + col instead of out + c * out_stride (channel_row)
    float *const *rows;
    long long col;
};

// ByteSampleConverter / SignedByteSampleConverter (J/source/tuner/... lookup tables: (b - 127) / 128.0f, b / 128.0f): both
// steps are exact in float, so converting on load gives the bits convert_kernel would have written
__device__ __forceinline__ float2 load_raw(const ChanParams &p, long long idx)
{
    const uchar2 b = __ldg(reinterpret_cast<const uchar2 *>(p.raw) + idx);
    const int vi = (int)(b.x ^ p.raw_flip) - p.raw_bias, vq = (int)(b.y ^ p.raw_flip) - p.raw_bias;
    return make_float2(__fmul_rn((float)vi, 0.0078125f), __fmul_rn((float)vq, 0.0078125f));
}

// sample idx of the virtual stream [state | in | zeros] the filter bank reads: the history (and leftover samples) the call
// starts from, its new samples, then zeros; state(i) and in(i) load sample i of the first two
template <class State, class In>
__device__ __forceinline__ float2 stream_sample(int idx, int state_len, int n_in, State state, In in)
{
    if (idx < state_len) return state(idx);
    idx -= state_len;
    return idx < n_in ? in(idx) : make_float2(0.0f, 0.0f);
}

template <bool RAW = false>
__device__ __forceinline__ float2 load_x(const ChanParams &p, int unit, int r)
{
    // unit 0 starts right after the history
    return stream_sample(p.H + unit * p.half + r, p.state_len, p.n_in, [&](int i) { return __ldg(p.state + i); },
                         [&](int i) { return RAW ? load_raw(p, i) : __ldg(p.in + i); });
}

__device__ __forceinline__ float2 cmul(float2 a, float2 w)
{
    // explicit FMA is fine here: the inverse DFT is compared at 1e-4 relative RMS, not bit-exactly
    return make_float2(fmaf(a.x, w.x, -a.y * w.y), fmaf(a.x, w.y, a.y * w.x));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 jmul(float2 a) { return make_float2(-a.y, a.x); }  // * (+j)

template <int NB, int TT, bool ROUTED>
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
            float *row = c < p.n_main ? channel_row<ROUTED>(p.out, p.out_stride, p.rows, p.col, c)
                                      : p.out2 + (size_t)(c - p.n_main) * p.out2_stride;
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
// (400 = 20 x 20, 800 = 32 x 25, 96 = 8 x 12, ... see kPfbRows).  One CTA per tile of NB consecutive blocks:
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
                const float2 pr = __ffma2_rn(x, make_float2(hA[t], hA[t]), nz);
                // (the Java's 0.0f + product differs from the product only in the sign of a zero)
                if (t == 0) accA[bl] = pr;
                else accA[bl] = __fadd2_rn(accA[bl], pr);
            }
            const int bm = pp + 1 + 2 * t;  // branch n + M/2: unit P = B - 1 - 2t
            if (bm >= 0 && bm < NB) {
                const float2 pr = __ffma2_rn(x, make_float2(hB[t], hB[t]), nz);
                if (t == 0) accB[bm] = pr;
                else accB[bm] = __fadd2_rn(accB[bm], pr);
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

template <int M, int R1, int R2, int NB, int TT, int NT, int MINB, bool RAW, bool ROUTED>
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
        for (int i = tid; i < p.next_len; i += NT)
            p.next_state[i] = stream_sample(p.consumed + i, p.state_len, p.n_in, [&](int j) { return p.state[j]; },
                                            [&](int j) { return RAW ? load_raw(p, j) : p.in[j]; });
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
                // bin k1 + R1 k2 is row k1 + R1 k2; routed rows are looked up one by one (channel_row)
                float *o = ROUTED ? nullptr : p.out + (size_t)k1 * p.out_stride + 2 * (size_t)(b0 + b);
                const size_t ostep = (size_t)R1 * p.out_stride;
                auto dst = [&](int k2) {
                    return ROUTED ? channel_row<true>(nullptr, 0, p.rows, p.col + 2 * (b0 + b), k1 + R1 * k2) : o;
                };
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
                        const float2 m = mix_complex(make_float2(__fmul_rn(a[k2].x, inv), __fmul_rn(a[k2].y, inv)), __ldg(zp));
                        *reinterpret_cast<float2 *>(dst(k2)) = make_float2(__fmul_rn(m.x, g), __fmul_rn(m.y, g));
                        if (!ROUTED) o += ostep;
                        zp += zstep;
                    }
                } else {
#pragma unroll
                    for (int k2 = 0; k2 < R2; k2++) {
                        // (1 / M, then the gain: two packed multiplies for four scalar ones)
                        const float2 v = __fmul2_rn(__fmul2_rn(a[k2], make_float2(inv, inv)), make_float2(g, g));
                        *reinterpret_cast<float2 *>(dst(k2)) = v;
                        if (!ROUTED) o += ostep;
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
                float *o = ROUTED ? nullptr : out + (size_t)row0 * p.out_stride;
                const size_t ostep = (size_t)ROWS * p.out_stride;
                const float2 *xr = X + bl * XS;
#pragma unroll 5
                for (int c = row0; c < M; c += ROWS) {
                    float2 v = xr[c];
                    v.x = __fmul_rn(__fmul_rn(v.x, inv_m), g);
                    v.y = __fmul_rn(__fmul_rn(v.y, inv_m), g);
                    *reinterpret_cast<float2 *>(ROUTED ? channel_row<true>(nullptr, 0, p.rows, p.col + 2 * b, c) : o) = v;
                    if (!ROUTED) o += ostep;
                }
            } else if (p.gain_exact) {
                for (int c = row0; c < p.n_sel; c += ROWS) {
                    const float g = __ldg(p.gain_f + c);
                    float2 v = X[bl * XS + __ldg(p.sel + c)];
                    v.x = __fmul_rn(__fmul_rn(v.x, inv_m), g);
                    v.y = __fmul_rn(__fmul_rn(v.y, inv_m), g);
                    float *row = c < p.n_main ? channel_row<ROUTED>(p.out, p.out_stride, p.rows, p.col, c)
                                              : p.out2 + (size_t)(c - p.n_main) * p.out2_stride;
                    *reinterpret_cast<float2 *>(row + 2 * (size_t)b) = v;
                }
            } else {
                for (int c = row0; c < p.n_sel; c += ROWS) {
                    const double g = __ldg(p.gain_d + c);
                    float2 v = X[bl * XS + __ldg(p.sel + c)];
                    v.x = __double2float_rn(__dmul_rn((double)__fmul_rn(v.x, inv_m), g));
                    v.y = __double2float_rn(__dmul_rn((double)__fmul_rn(v.y, inv_m), g));
                    float *row = c < p.n_main ? channel_row<ROUTED>(p.out, p.out_stride, p.rows, p.col, c)
                                              : p.out2 + (size_t)(c - p.n_main) * p.out2_stride;
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

// new_state[i] = S[consumed + i], S = [state | in | zeros]
__global__ void save_state_kernel(const float2 *state, int state_len, const float2 *in, int n_in, int consumed,
                                  float2 *new_state, int new_len)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < new_len; i += gridDim.x * blockDim.x)
        new_state[i] = stream_sample(consumed + i, state_len, n_in, [&](int j) { return state[j]; }, [&](int j) { return in[j]; });
}

// L2 read-ahead distance of pfb2_kernel in blocks: two 8-block tiles for each of the 148 SMs of a B200, the measured
// optimum (half a wave of the M = 400 kernel at 4 CTAs per SM, two thirds of one of the M = 800 kernel at 3)
constexpr int kPfbPrefetchBlocks = 148 * 8 * 2;

// One pfb2_kernel shape: M = R1 x R2 channels, NB blocks per tile, NT threads, at least MINB CTAs per SM.  f32 launches
// the instance for float input; raw, if there is one, the instance that reads 8-bit tuner samples and converts on load.
// Each comes as [0] contiguous rows and [1] routed rows (ChanParams::rows).
using PfbLauncher = sdrgpu_status (*)(const sdrgpu_channelizer *h, const ChanParams &p);
struct PfbRow {
    int M, R1, R2, NB, NT, MINB;
    PfbLauncher f32[2], raw[2];
};

}  // namespace

// ---------------------------------------------------------------------------------------------------- handle
struct sdrgpu_channelizer {
    int device = 0;
    int M = 0, T = 0, half = 0, H = 0, NB = 16;
    int max_in_complex = 0, max_blocks = 0;
    int leftover = 0, parity0 = 0;
    bool throttled = false;   // chan_set_throttled: the pipeline is overlapping this launch with the demodulator
    // chan_convert leaves 8-bit tuner samples unconverted for chan_enqueue when the filter bank converts them on load (no
    // float copy of the input in HBM, converts_on_load); otherwise convert_kernel converts them first
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
    const PfbRow *fast = nullptr;   // the pfb2_kernel row of this channel count (nullptr: pfb_ifft_kernel)
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
    ChanOutputs outputs;               // two-bin and frequency-corrected channels (outputs.cu)
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

// the filter bank's rows and gains for the output stage's rows `r`, and the store paths they allow
sdrgpu_status upload_rows(sdrgpu_channelizer *h, const OutputRows &r)
{
    const int n = (int)h->channels.size(), rows = (int)r.sel.size();
    std::vector<float> gf(rows);
    int exact = 1;
    for (int i = 0; i < rows; i++) {
        gf[i] = (float)r.gain[i];
        if ((double)gf[i] != r.gain[i]) exact = 0;
    }
    cudaFree(h->d_sel);
    cudaFree(h->d_gain_f);
    cudaFree(h->d_gain_d);
    h->d_sel = nullptr;
    h->d_gain_f = nullptr;
    h->d_gain_d = nullptr;
    SDRGPU_CUDA(cudaMalloc(&h->d_sel, sizeof(int) * (size_t)rows));
    SDRGPU_CUDA(cudaMalloc(&h->d_gain_f, sizeof(float) * (size_t)rows));
    SDRGPU_CUDA(cudaMalloc(&h->d_gain_d, sizeof(double) * (size_t)rows));
    SDRGPU_CUDA(cudaMemcpy(h->d_sel, r.sel.data(), sizeof(int) * (size_t)rows, cudaMemcpyHostToDevice));
    SDRGPU_CUDA(cudaMemcpy(h->d_gain_f, gf.data(), sizeof(float) * (size_t)rows, cudaMemcpyHostToDevice));
    SDRGPU_CUDA(cudaMemcpy(h->d_gain_d, r.gain.data(), sizeof(double) * (size_t)rows, cudaMemcpyHostToDevice));
    h->mix_identity = r.mix_identity;
    h->mix_gain = r.mix_gain;
    h->n_sel = n;
    h->n_rows = rows;
    h->gain_exact = exact;
    h->identity = exact && n == h->M && h->outputs.n_post == 0 && h->outputs.n_mix == 0;
    for (int i = 0; i < n && h->identity; i++)
        if (r.sel[i] != i || gf[i] != gf[0]) h->identity = 0;
    h->gain_uniform = n > 0 ? gf[0] : 0.0f;
    return SDRGPU_OK;
}

sdrgpu_status upload_selection(sdrgpu_channelizer *h)
{
    OutputRows r;
    SDRGPU_TRY(outputs_select(h->outputs, h->channels, h->M, h->sample_rate, h->max_blocks, &r));
    return upload_rows(h, r);
}

template <int M, int R1, int R2, int NB, int TT, int NT, int MINB, bool RAW, bool ROUTED>
sdrgpu_status launch_pfb2(const sdrgpu_channelizer *h, const ChanParams &p)
{
    using L = Pfb2Layout<M, R1, R2, NB, TT, NT>;
    auto kernel = pfb2_kernel<M, R1, R2, NB, TT, NT, MINB, RAW, ROUTED>;
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

template <int NB, int TT, bool ROUTED>
sdrgpu_status launch_pfb(const sdrgpu_channelizer *h, const ChanParams &p, int grid)
{
    auto kernel = pfb_ifft_kernel<NB, TT, ROUTED>;
    SDRGPU_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_bytes));
    kernel<<<grid, kThreads, h->smem_bytes, h->stream>>>(p);
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    return SDRGPU_OK;
}

template <int M, int R1, int R2, int NB, int NT, int MINB, bool RAW>
constexpr PfbRow pfb_row()
{
    PfbRow row{M, R1, R2, NB, NT, MINB, {launch_pfb2<M, R1, R2, NB, 9, NT, MINB, false, false>,
                                         launch_pfb2<M, R1, R2, NB, 9, NT, MINB, false, true>}, {nullptr, nullptr}};
    if constexpr (RAW) {
        row.raw[0] = launch_pfb2<M, R1, R2, NB, 9, NT, MINB, true, false>;
        row.raw[1] = launch_pfb2<M, R1, R2, NB, 9, NT, MINB, true, true>;
    }
    return row;
}

// The pfb2_kernel instances: the channel counts of the common tuner rates (25 kHz channels: 2 / 2.4 / 2.5 / 3 / 4 / 5 / 6 /
// 8 / 10 / 16 / 20 MS/s) with the reference's 9 taps per channel.  Tile shapes measured on a B200 (profiles/): M = 400 runs
// best as 8-block tiles, 200 threads, 4 CTAs per SM; M = 800 as 8-block tiles, 256 threads, 3 CTAs per SM.  8-block tiles
// store a default selection straight from step B (and mix the oscillators in there, fused_mix in chan_enqueue).
constexpr PfbRow kPfbRows[] = {
    pfb_row<400, 20, 20, 8, 200, 4, true>(),
    pfb_row<800, 32, 25, 8, 256, 3, true>(),
    pfb_row<96, 8, 12, 16, 192, 2, false>(),
    pfb_row<640, 32, 20, 8, 320, 2, false>(),
    pfb_row<320, 16, 20, 8, 160, 4, false>(),
    pfb_row<240, 12, 20, 8, 160, 4, false>(),
    pfb_row<200, 10, 20, 8, 160, 4, false>(),
    pfb_row<160, 8, 20, 8, 160, 4, false>(),
    pfb_row<120, 10, 12, 16, 192, 2, false>(),
    pfb_row<100, 10, 10, 16, 160, 2, false>(),
    pfb_row<80, 8, 10, 16, 160, 2, false>(),
};

// The filter bank and inverse DFT of one call: the handle's pfb2_kernel row (its 8-bit instance if raw), else
// pfb_ifft_kernel.
sdrgpu_status pfb_launch(const sdrgpu_channelizer *h, const ChanParams &p, bool raw)
{
    const bool routed = p.rows != nullptr;
    if (h->fast) return (raw ? h->fast->raw : h->fast->f32)[routed](h, p);
    const int grid = (p.n_blocks + h->NB - 1) / h->NB;
    if (routed) {
        if (h->NB == 16) return h->T == 9 ? launch_pfb<16, 9, true>(h, p, grid) : launch_pfb<16, 0, true>(h, p, grid);
        return h->T == 9 ? launch_pfb<8, 9, true>(h, p, grid) : launch_pfb<8, 0, true>(h, p, grid);
    }
    if (h->NB == 16) return h->T == 9 ? launch_pfb<16, 9, false>(h, p, grid) : launch_pfb<16, 0, false>(h, p, grid);
    return h->T == 9 ? launch_pfb<8, 9, false>(h, p, grid) : launch_pfb<8, 0, false>(h, p, grid);
}

// whether the filter bank reads 8-bit tuner samples as they are
bool converts_on_load(const sdrgpu_channelizer *h) { return h->fast && h->fast->raw[0]; }

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
                                   int layout, int *n_blocks_out, float *const *rows, long long col)
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
    const bool fuse_convert = raw && n_blocks > 0 && converts_on_load(h);
    if (raw && !fuse_convert) launch_convert(h, raw, const_cast<float2 *>(d_in), n_in);
    ChanOutputs &o = h->outputs;
    // checked before anything is launched or the framing state advances: a failing call leaves the handle as it was
    if (n_blocks > 0 && (o.n_mix > 0 || o.n_post > 0)) {
        // The reference rotates every channel's mixer for every buffer; the results layout has no per-channel rows to
        // mix, and skipping the oscillators would leave them out of step with the sample stream for later calls.
        if (layout != SDRGPU_LAYOUT_CHANNELS)
            return fail(SDRGPU_ERR_BAD_STATE, "two-bin / frequency-corrected channels are selected: use SDRGPU_LAYOUT_CHANNELS");
        if (o.n_mix > 0 && n_blocks > o.osc_ring_len)
            return fail(SDRGPU_ERR_OVERFLOW, "%d blocks exceed the oscillator look-ahead", n_blocks);
    }
    // Frequency-corrected one-bin channels: the oscillator values come from the look-ahead rings (osc_produce_kernel on a
    // side stream).  When every bin is such a channel and the pfb2_kernel instance stores the rows straight from step B
    // (8-block tiles), it multiplies them in there (no separate pass over the channel streams); otherwise the rows leave
    // the kernel at gain 1 and osc_mix_kernel finishes them.
    const bool fused_mix = o.n_mix > 0 && h->mix_identity && h->fast && h->fast->NB == 8 && layout == SDRGPU_LAYOUT_CHANNELS &&
                           n_blocks > 0;
    if (n_blocks > 0) {
        ChanParams p{};
        p.neg_zero = -0.0f;
        p.rows = rows;
        p.col = col;
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
        p.out2 = o.d_out2;
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
        p.osc_ring_len = o.osc_ring_len;
        if (fused_mix) SDRGPU_TRY(outputs_before(o, n_blocks, h->stream, &p.osc, &p.osc_start));
        p.prefetch_blocks = kPfbPrefetchBlocks;
        p.gain_uniform = fused_mix ? h->mix_gain : h->gain_uniform;
        p.inv_m = 1.0f / (float)h->M;
        p.n_factors = (int)h->factors.size();
        for (int i = 0; i < p.n_factors; i++) {
            p.factors[i] = h->factors[i];
            p.magic_s[i] = h->magic[i];
        }
        if (h->fast && n_in > 0) {
            p.next_state = next;
            p.next_len = new_len;
            p.consumed = consumed;
            state_saved = true;
        }
        h->timer.begin(h->stream);
        const sdrgpu_status st = pfb_launch(h, p, fuse_convert);
        h->timer.end(h->stream);
        SDRGPU_TRY(st);
        if (layout == SDRGPU_LAYOUT_CHANNELS) SDRGPU_TRY(outputs_after(o, d_out, stride, n_blocks, fused_mix, h->stream, rows, col));
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
        if (eight_bit && converts_on_load(h)) {
            h->defer_src = src + cb * first;
            h->defer_dst = h->d_in + first;
            h->defer_n = n;
        } else {
            launch_convert(h, src + cb * first, h->d_in + first, n);
        }
    }
    return h->d_in + first;
}
sdrgpu_status sdrgpu::chan_osc_ahead(sdrgpu_channelizer *h) { return outputs_ahead(h->outputs, h->stream); }

cudaStream_t sdrgpu::chan_osc_stream(const sdrgpu_channelizer *h) { return h->outputs.n_mix > 0 ? h->outputs.osc_stream : nullptr; }

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
    if (h->T == 9)
        for (const PfbRow &row : kPfbRows)
            if (row.M == M) h->fast = &row;
    if (h->fast) {
        std::vector<float2> tw2((size_t)M);
        for (int k1 = 0; k1 < h->fast->R1; k1++)
            for (int n2 = 0; n2 < h->fast->R2; n2++) {
                const double a = 2.0 * 3.14159265358979323846 * (double)((long long)k1 * n2 % M) / (double)M;
                tw2[(size_t)k1 * h->fast->R2 + n2] = make_float2((float)cos(a), (float)sin(a));
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
    sdrgpu::outputs_destroy(h->outputs);
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
    if (changed && (h->outputs.n_mix > 0 || h->outputs.n_post > 0)) {
        SDRGPU_CUDA(cudaSetDevice(h->device));
        SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
        return upload_selection(h);
    }
    return SDRGPU_OK;
}

namespace {

// the bins of a selection are in range; two-bin and frequency-corrected channels need the sample rate
sdrgpu_status check_channels(const sdrgpu_channelizer *h, const sdrgpu_output_channel *channels, int n_channels,
                             bool *any_two)
{
    bool any_special = false;
    *any_two = false;
    for (int i = 0; i < n_channels; i++) {
        if (channels[i].bin1 < 0 || channels[i].bin1 >= h->M)
            return fail(SDRGPU_ERR_INVALID_ARG, "Channel [%d] is not valid -- max channel is %d", channels[i].bin1, h->M);
        if (channels[i].bin2 >= h->M)
            return fail(SDRGPU_ERR_INVALID_ARG, "Channel [%d] is not valid -- max channel is %d", channels[i].bin2, h->M);
        *any_two |= channels[i].bin2 >= 0;
        any_special |= channels[i].bin2 >= 0 || channels[i].frequency_offset_hz != 0;
    }
    if (any_special && !(h->sample_rate > 0.0))
        return fail(SDRGPU_ERR_BAD_STATE, "two-bin / frequency-corrected channels need sdrgpu_chan_set_sample_rate first");
    return SDRGPU_OK;
}

sdrgpu_status parse_synthesis_filter(const float *synthesis_filter, int n_synthesis_taps, SynthFilter *synth)
{
    if (!synthesis_filter || n_synthesis_taps < 2)
        return fail(SDRGPU_ERR_INVALID_ARG, "two-bin channels need the synthesis filter (getSincM2Synthesizer)");
    // TwoChannelSynthesizerM2.init (:74-88): tapsPerChannel = ceil(filter.length / 2) with integer division; the
    // I/Q-duplicated filter has 2 * tapsPerChannel * 2 entries
    const int entries = n_synthesis_taps / 2;
    if (entries > kMaxSynthEntries)
        return fail(SDRGPU_ERR_INVALID_ARG, "synthesis filter longer than %d taps", 2 * kMaxSynthEntries);
    std::memset(synth, 0, sizeof(*synth));
    synth->entries = entries;
    int fp = 0;
    for (int cp = 0; cp < n_synthesis_taps && fp + 1 < 4 * entries; cp++) {
        synth->f[fp++] = synthesis_filter[cp];
        synth->f[fp++] = synthesis_filter[cp];
    }
    return SDRGPU_OK;
}

}  // namespace

sdrgpu_status sdrgpu_chan_select(sdrgpu_channelizer *h, const sdrgpu_output_channel *channels, int n_channels,
                                 const float *synthesis_filter, int n_synthesis_taps)
{
    if (!h || !channels || n_channels <= 0) return fail(SDRGPU_ERR_INVALID_ARG, "NULL / empty selection");
    bool any_two = false;
    SDRGPU_TRY(check_channels(h, channels, n_channels, &any_two));
    if (any_two) SDRGPU_TRY(parse_synthesis_filter(synthesis_filter, n_synthesis_taps, &h->outputs.synth));
    SDRGPU_CUDA(cudaStreamSynchronize(h->stream));
    h->channels.assign(channels, channels + n_channels);
    return upload_selection(h);
}

sdrgpu_status sdrgpu_chan_update_selection(sdrgpu_channelizer *h, const sdrgpu_output_channel *channels,
                                           const int *previous, int n_channels, const float *synthesis_filter,
                                           int n_synthesis_taps)
{
    if (!h || !channels || !previous || n_channels <= 0) return fail(SDRGPU_ERR_INVALID_ARG, "NULL / empty selection");
    bool any_two = false, kept_two = false;
    SDRGPU_TRY(check_channels(h, channels, n_channels, &any_two));
    const int n_old = (int)h->channels.size();
    std::vector<char> named((size_t)n_old, 0);
    for (int i = 0; i < n_channels; i++) {
        const int p = previous[i];
        if (p < -1 || p >= n_old)
            return fail(SDRGPU_ERR_INVALID_ARG, "entry %d continues channel %d of a selection of %d channels", i, p, n_old);
        if (p < 0) continue;
        if (named[(size_t)p]) return fail(SDRGPU_ERR_INVALID_ARG, "channel %d is continued twice", p);
        named[(size_t)p] = 1;
        // OneChannelOutputProcessor / TwoChannelOutputProcessor take the gain and the bin count at creation
        const sdrgpu_output_channel &was = h->channels[(size_t)p];
        if ((was.bin2 >= 0) != (channels[i].bin2 >= 0))
            return fail(SDRGPU_ERR_INVALID_ARG, "entry %d changes the bin count of channel %d: make it a new channel", i, p);
        if (was.gain != channels[i].gain)
            return fail(SDRGPU_ERR_INVALID_ARG, "entry %d changes the gain of channel %d: make it a new channel", i, p);
        kept_two |= was.bin2 >= 0;
    }
    SynthFilter synth = h->outputs.synth;
    if (synthesis_filter) {
        if (kept_two)
            return fail(SDRGPU_ERR_INVALID_ARG, "a new synthesis filter restarts the two-bin channels: sdrgpu_chan_select");
        SDRGPU_TRY(parse_synthesis_filter(synthesis_filter, n_synthesis_taps, &synth));
    } else if (any_two && synth.entries == 0) {
        return fail(SDRGPU_ERR_INVALID_ARG, "two-bin channels need the synthesis filter (getSincM2Synthesizer)");
    }
    SDRGPU_CUDA(cudaSetDevice(h->device));
    const std::vector<sdrgpu_output_channel> next(channels, channels + n_channels);
    OutputRows r;
    // outputs_update waits for the calls in flight, which read the current filter, before anything changes
    SDRGPU_TRY(outputs_update(h->outputs, h->channels, next, std::vector<int>(previous, previous + n_channels), h->M,
                              h->sample_rate, h->stream, &r));
    h->outputs.synth = synth;
    h->channels = next;
    return upload_rows(h, r);
}

sdrgpu_status sdrgpu_chan_set_frequency_offsets(sdrgpu_channelizer *h, const int *channels, const long long *offsets_hz, int n)
{
    if (!h || !channels || !offsets_hz || n <= 0) return fail(SDRGPU_ERR_INVALID_ARG, "NULL / empty argument");
    const int n_sel = (int)h->channels.size();
    std::vector<char> seen((size_t)n_sel, 0);
    bool any_offset = false;
    for (int i = 0; i < n; i++) {
        if (channels[i] < 0 || channels[i] >= n_sel)
            return fail(SDRGPU_ERR_INVALID_ARG, "channel %d is not in the selection of %d channels", channels[i], n_sel);
        if (seen[(size_t)channels[i]]) return fail(SDRGPU_ERR_INVALID_ARG, "channel %d is listed twice", channels[i]);
        seen[(size_t)channels[i]] = 1;
        any_offset |= offsets_hz[i] != 0;
    }
    if (any_offset && !(h->sample_rate > 0.0))
        return fail(SDRGPU_ERR_BAD_STATE, "frequency-corrected channels need sdrgpu_chan_set_sample_rate first");
    // a repeat of a channel's offset changes nothing (Oscillator.update computes the same angle)
    std::vector<sdrgpu_output_channel> next = h->channels;
    std::vector<int> changed;
    for (int i = 0; i < n; i++)
        if (next[(size_t)channels[i]].frequency_offset_hz != offsets_hz[i]) {
            next[(size_t)channels[i]].frequency_offset_hz = offsets_hz[i];
            changed.push_back(channels[i]);
        }
    if (changed.empty()) return SDRGPU_OK;
    SDRGPU_CUDA(cudaSetDevice(h->device));
    OutputRows r;
    bool rows_changed = false;
    SDRGPU_TRY(outputs_set_offsets(h->outputs, h->channels, next, changed, h->M, h->sample_rate, h->stream, &r,
                                   &rows_changed));
    h->channels = next;
    if (rows_changed) SDRGPU_TRY(upload_rows(h, r));
    return SDRGPU_OK;
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
