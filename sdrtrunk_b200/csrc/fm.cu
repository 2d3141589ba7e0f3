// The FM stage of a bank (fm.cuh): power squelch and FM discriminator, and the fused NBFM front end.
//
// Replaces, per channel (J/ = src/main/java/io/github/dsheirer/):
//   FMDemodulator / SquelchingFMDemodulator            J/dsp/fm/FMDemodulator.java:62-96, SquelchingFMDemodulator.java:63-101
//   PowerSquelch.process                               J/dsp/squelch/PowerSquelch.java:88-159
//   NBFMDecoder.receive (decimation, FIR, squelch, FM) J/module/decode/nbfm/NBFMDecoder.java:129-181
//
// Arithmetic contract: float ops are separately rounded (-fmad=false, __f*_rn) exactly where the Java has separate
// * and +; fmaf in tap order where the Java calls Math.fma; the squelch's IIR and the discriminator's atan in double,
// as the Java does.
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "fm.cuh"
#include "tma.cuh"

using namespace sdrgpu;

namespace {

// ---------------------------------------------------------------------------------------------------------------
// FM discriminator.  Squelch gate: sequential per channel (double one-pole IIR + ramp state machine); the atan
// discriminator itself is data parallel.
// ---------------------------------------------------------------------------------------------------------------

// PowerSquelch's ramp state machine for one sample (state: SquelchState::state); true where SquelchingFMDemodulator
// demodulates the sample (UNMUTE or DECAY)
__device__ __forceinline__ bool squelch_step(int &state, int &ramp_count, bool mute, int ramp)
{
    // (on copies: updating the references in place costs the fused kernel's chain an instruction)
    int s = state, r = ramp_count;
    switch (s) {
        case 2:  // MUTE
            if (!mute) {
                if (ramp > 0) { s = 0; r++; } else { s = 3; }
            }
            break;
        case 0:  // ATTACK
            if (r >= ramp) s = 3; else r++;
            break;
        case 1:  // DECAY
            if (r <= 0) s = 2; else r--;
            break;
        default:  // UNMUTE
            if (mute) {
                if (ramp > 0) { s = 1; r--; } else { s = 2; }
            }
            break;
    }
    state = s;
    ramp_count = r;
    return s == 3 || s == 1;
}

// one thread per channel: writes gate[n] = 1 where SquelchingFMDemodulator demodulates (UNMUTE or DECAY) and, with
// `status`, one squelch status byte per buffer_len samples.  Within the ramp machine the state changes
// (PowerSquelch.mSquelchChanged) exactly where the gate flips, so a buffer's CHANGED bit is "the gate has an edge in
// it"; the gate in front of the call's first sample is that of the state it starts from.
__global__ void squelch_gate_kernel(const float2 *__restrict__ in, long long in_stride, int n, SquelchState *states,
                                    uint8_t *__restrict__ gate, long long gate_stride, double alpha,
                                    const double *__restrict__ thresholds, int ramp, uint8_t *__restrict__ status,
                                    long long status_stride, int buffer_len, int n_channels)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_channels) return;
    SquelchState st = states[ch];
    const double one_minus = 1.0 - alpha, threshold = thresholds[ch];
    const float2 *x = in + (size_t)ch * in_stride;
    uint8_t *g = gate + (size_t)ch * gate_stride;
    uint8_t *rep = status ? status + (size_t)ch * status_stride : nullptr;
    bool on_before = st.state & 1, changed = false;
    int left = buffer_len;
    for (int k = 0; k < n; k++) {
        const float2 s = x[k];
        const double i = (double)s.x, q = (double)s.y;
        const double power_in = __dadd_rn(__dmul_rn(i, i), __dmul_rn(q, q));
        st.output = __dadd_rn(__dmul_rn(st.output, one_minus), __dmul_rn(alpha, power_in));
        const bool on = squelch_step(st.state, st.ramp_count, st.output < threshold, ramp);
        g[k] = on ? 1 : 0;
        if (rep) {
            changed |= on != on_before;
            on_before = on;
            if (--left == 0) {
                *rep++ = (uint8_t)(st.state | (changed ? SDRGPU_SQUELCH_CHANGED : 0));
                changed = false;
                left = buffer_len;
            }
        }
    }
    states[ch].output = st.output;
    states[ch].state = st.state;
    states[ch].ramp_count = st.ramp_count;
}

__device__ __forceinline__ float fm_angle(float ci, float cq, float pi_, float pq, float gain)
{
    // FMDemodulator.demodulate: float products / sums, then double
    const double inphase = (double)__fsub_rn(__fmul_rn(ci, pi_), __fmul_rn(cq, -pq));
    const double quadrature = (double)__fadd_rn(__fmul_rn(cq, pi_), __fmul_rn(ci, -pq));
    double angle = 0.0;
    if (inphase != 0) {
        const double denominator = __ddiv_rn(1.0, inphase);
        angle = atan(__dmul_rn(quadrature, denominator));
    }
    return __double2float_rn(__dmul_rn(angle, (double)gain));
}

// gate == nullptr: plain FMDemodulator (previous sample = n-1).  With a gate, the previous sample is the most
// recent gated one (the demodulator state is not updated while muted, SquelchingFMDemodulator.java:80-87).
__global__ void fm_kernel(const float2 *__restrict__ in, long long in_stride, int n, const uint8_t *__restrict__ gate,
                          long long gate_stride, const SquelchState *__restrict__ states, float gain,
                          float *__restrict__ out, long long out_stride)
{
    const int ch = blockIdx.y;
    const float2 *x = in + (size_t)ch * in_stride;
    const uint8_t *g = gate ? gate + (size_t)ch * gate_stride : nullptr;
    float *y = out + (size_t)ch * out_stride;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        if (g && !g[k]) {
            y[k] = 0.0f;
            continue;
        }
        int p = k - 1;
        if (g)
            while (p >= 0 && !g[p]) p--;
        float pi_, pq;
        if (p >= 0) {
            pi_ = x[p].x;
            pq = x[p].y;
        } else {
            pi_ = states[ch].prev_i;
            pq = states[ch].prev_q;
        }
        const float2 s = x[k];
        y[k] = fm_angle(s.x, s.y, pi_, pq, gain);
    }
}

// after fm_kernel: remember the last demodulated sample of every channel
__global__ void fm_carry_kernel(const float2 *__restrict__ in, long long in_stride, int n, const uint8_t *__restrict__ gate,
                                long long gate_stride, SquelchState *states, int n_channels)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_channels) return;
    const float2 *x = in + (size_t)ch * in_stride;
    const uint8_t *g = gate ? gate + (size_t)ch * gate_stride : nullptr;
    int p = n - 1;
    if (g)
        while (p >= 0 && !g[p]) p--;
    if (p >= 0) {
        states[ch].prev_i = x[p].x;
        states[ch].prev_q = x[p].y;
    }
}

// sdrgpu_bank_set_squelch_threshold: a launch rather than a copy, so that the value is ordered behind the calls already
// enqueued without a host buffer that has to outlive them
__global__ void set_threshold_kernel(double *thresholds, int n, double value)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) thresholds[i] = value;
}

// ---------------------------------------------------------------------------------------------------------------
// nbfm_fused_kernel: the whole NBFM front end of one channel in ONE launch (NBFMDecoder.receive,
// J/module/decode/nbfm/NBFMDecoder.java:129-181):
//   half-band decimation cascade (ComplexHalfBandDecimationFilter.java:66-123, up to kMaxFusedStages stages)
//   -> complex FIR (ComplexFIRFilter2.java:112-129, fma chain; I / Q rails share a packed FFMA2)
//   -> power squelch (PowerSquelch.java:88-159: double one-pole IIR + ramp state machine, serial)
//   -> FM discriminator epilogue (FMDemodulator.java:62-96: conjugate product with the previous demodulated sample, atan)
// One CTA per channel walks its row in tiles of `tile_out` output samples.  The input window of a tile -- regular and
// contiguous -- is fetched by cp.async.bulk (TMA engine) while the tile before it is computed; an mbarrier counts the
// bytes in (decimating banks: one window buffer, de-interleaved into even / odd sample planes as soon as it has arrived,
// the next window's copy issued right behind that; no decimation: a double buffer, the FIR reads the window itself).  Intermediate samples never leave shared memory: HBM traffic is
// the 8 B / input sample read + 4 B / output sample written.  Every filter is a pure function of the input stream, so the
// samples a tile's first outputs need from before the tile (N - 1 decimated samples, each L - 1 raw ones) are recomputed
// from `hist0` raw samples of history instead of being carried as per-stage state: bit-identical, and no carry kernels.
// The squelch's IIR is a two-operation dependent chain per output sample on one thread; the products it consumes are
// computed by all threads beforehand, and the other channels' CTAs fill the SM while it runs.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kMaxFusedStages = 3;
constexpr int kNbfmThreads = 128;
constexpr int kNbfmFilterThreads = 96;   // warps 0 .. 2 filter; warp 3 runs the serial squelch chain a tile behind them

struct NbfmParams {
    const float2 *hist;        // [C][hist0] raw samples in front of the new ones
    long long hist_stride;
    const float2 *in;          // [C][n_new] new samples
    long long in_stride;
    float2 *hist_out;          // [C][hist0] history for the next call (the other half of a ping-pong)
    long long hist_out_stride;
    int n_new, hist0;
    int n_stages;
    int n_fir;
    float fir_gain;
    int tile_out;              // final-rate outputs per tile
    int window_cap;            // float2 per raw window buffer (16-byte multiple)
    int use_bulk;              // rows are 16-byte aligned: windows arrive by cp.async.bulk
    int cap_e0, cap_o0, cap_e1, cap_o1, cap_z;   // float2 per plane / FIR input buffer (decimating variant, nbfm_fused_layout)
    float neg_zero;            // -0.0f, as a run-time value (see the half-band stages)
    int squelch;               // SquelchingFMDemodulator (else FMDemodulator: every sample demodulated)
    double alpha;
    const double *thresholds;  // [C]
    int ramp;
    float fm_gain;
    SquelchState *sq;
    float *out;                // [C][n_new / 2^n_stages] demodulated floats, may be null
    long long out_stride;
    uint8_t *status;           // kStatus: [C][status_stride] one squelch status byte per buffer_out outputs
    long long status_stride;
    int buffer_out;
    int n_channels;
};

struct NbfmStageTaps {
    HalfBandTaps stage[kMaxFusedStages];
};

// Shared-memory layout of the skewed buffers: float2 index p lives at p + 2 (p >> 2), i.e. 16 bytes of padding behind every 32,
// so that threads which own FOUR consecutive samples each (lane stride 32 bytes) fetch them with LDS.128 at a lane stride of
// 48 bytes: the eight lanes of a quarter warp then cover all 32 banks.  (r3a ncu: 264 M of the kernel's 486 M shared-memory
// wavefronts were bank conflicts -- LDS.64 at lane strides of 16 and 32 bytes -- and the LSU data pipe was 71 % busy.)
__host__ __device__ inline int nbfm_skew(int p) { return p + 2 * (p >> 2); }

// decimating variant (n_stages >= 1):
//   raw[window_cap] | E0 (skewed) | O0 | E1 (skewed) | O1 | Z (skewed) | filt[2][tile_out] | pw[2][tile_out] | gate bits[2][..]
// E / O = even- / odd-indexed samples of a half-band stage's input (the stage only multiplies even ones; the odd plane
// feeds its centre tap); Z = the last stage's output = the FIR's input.
// no decimation: raw[2][window_cap] | filt | pw | gate bits (the FIR reads the raw window).
inline void nbfm_fused_layout(NbfmParams &q, int first_stage_outputs)
{
    q.cap_e0 = q.cap_o0 = q.cap_e1 = q.cap_o1 = q.cap_z = 0;
    if (q.n_stages < 1) return;
    const int in0 = (1 << q.n_stages) * q.tile_out + q.hist0;
    q.cap_o0 = (in0 / 2 + 16) & ~1;
    q.cap_e0 = (nbfm_skew(in0 / 2 + 16) + 3) & ~1;
    if (q.n_stages >= 2) {
        q.cap_o1 = (first_stage_outputs / 2 + 16) & ~1;
        q.cap_e1 = (nbfm_skew(first_stage_outputs / 2 + 16) + 3) & ~1;
    }
    q.cap_z = (nbfm_skew(first_stage_outputs + 24) + 3) & ~1;
}

inline size_t nbfm_fused_smem(const NbfmParams &q)
{
    size_t bytes = sizeof(float2) * (q.n_stages >= 1 ? 1 : 2) * (size_t)q.window_cap;
    bytes += sizeof(float2) * (size_t)(q.cap_e0 + q.cap_o0 + q.cap_e1 + q.cap_o1 + q.cap_z);
    bytes += 2 * (sizeof(float2) * (size_t)q.tile_out + sizeof(double) * (size_t)q.tile_out + sizeof(uint32_t) * (size_t)(q.tile_out / 32 + 1));
    return (bytes + 15) & ~(size_t)15;
}

// kStatus: the chain thread also writes one squelch status byte per assembler buffer (p.status); a separate instance, so
// that banks which do not ask for statuses run the chain without the bookkeeping
template <bool kDecim, bool kStatus>
__global__ void __launch_bounds__(kNbfmThreads, 8)
nbfm_fused_kernel(const __grid_constant__ NbfmParams p, const __grid_constant__ NbfmStageTaps taps, const __grid_constant__ FirTaps fir)
{
    extern __shared__ __align__(16) unsigned char nbfm_smem[];
    __shared__ __align__(8) uint64_t bars[2];
    __shared__ float s_prev[2];          // FMDemodulator.mPreviousI / Q carried from tile to tile
    __shared__ double s_threshold;       // this channel's squelch threshold (read by the chain thread once per tile)
    __shared__ __align__(16) float hs[kMaxFirTaps];
    const int tid = threadIdx.x, c = blockIdx.x;
    const int S = p.n_stages, d = 1 << S, T = p.tile_out, N = p.n_fir;
    const int n_out_total = p.n_new >> S;
    const int n_tiles = (n_out_total + T - 1) / T;
    float2 *raw0 = reinterpret_cast<float2 *>(nbfm_smem);
    float2 *raw1 = raw0 + (kDecim ? 0 : p.window_cap);   // decimating variant: one window buffer (it is de-interleaved at once)
    float2 *pe0 = raw1 + p.window_cap;   // planes of the first stage's input (and of the third's)
    float2 *po0 = pe0 + p.cap_e0;
    float2 *pe1 = po0 + p.cap_o0;        // planes of the second stage's input
    float2 *po1 = pe1 + p.cap_e1;
    float2 *zs = po1 + p.cap_o1;         // the FIR's input (skewed)
    float2 *filt = zs + p.cap_z;         // [2][T]: tile t in half t & 1
    double *pw = reinterpret_cast<double *>(filt + 2 * T);              // [2][T]
    uint32_t *gate = reinterpret_cast<uint32_t *>(pw + 2 * T);          // [2][T / 32 + 1]: bit k & 31 of word k >> 5: sample k is demodulated
    const int gate_words = T / 32 + 1;

    const float2 *hist = p.hist + (size_t)c * p.hist_stride;
    const float2 *in = p.in + (size_t)c * p.in_stride;
    const int KP = fir_padded_taps(N);
    for (int k = tid; k < KP; k += kNbfmThreads) hs[k] = k < N ? fir.h[k] : 0.0f;
    SquelchState st = p.sq[c];
    if (tid == 0) {
        s_prev[0] = st.prev_i;
        s_prev[1] = st.prev_q;
        if (p.squelch) s_threshold = p.thresholds[c];
    }
    // kStatus: the output index that ends the current assembler buffer, whether the gate has had an edge in it so far,
    // and where its status byte goes
    int buffer_end = p.buffer_out - 1;
    bool changed = false;
    uint8_t *status_at = kStatus ? p.status + (size_t)c * p.status_stride : nullptr;

    // raw window of tile t: stream samples [t d T - hist0, t d T + d T_t); negative indices are history
    auto tile_outputs = [&](int t) { return min(T, n_out_total - t * T); };
    auto issue = [&](int t) {   // one thread: arm the barrier, start the copies
        float2 *dst = (t & 1) ? raw1 : raw0;
        const int n_in = d * tile_outputs(t);
        uint64_t *bar = &bars[kDecim ? 0 : (t & 1)];
        if (t == 0) {
            sdrgpu::tma::mbar_arrive_expect_tx(bar, (uint32_t)(sizeof(float2) * (size_t)(p.hist0 + n_in)));
            if (p.hist0 > 0) sdrgpu::tma::bulk_load(dst, hist, (uint32_t)(sizeof(float2) * (size_t)p.hist0), bar);
            sdrgpu::tma::bulk_load(dst + p.hist0, in, (uint32_t)(sizeof(float2) * (size_t)n_in), bar);
        } else {
            sdrgpu::tma::mbar_arrive_expect_tx(bar, (uint32_t)(sizeof(float2) * (size_t)(p.hist0 + n_in)));
            sdrgpu::tma::bulk_load(dst, in + ((size_t)t * d * T - p.hist0), (uint32_t)(sizeof(float2) * (size_t)(p.hist0 + n_in)), bar);
        }
    };
    if (p.use_bulk) {
        if (tid == 0) {
            sdrgpu::tma::mbar_init(&bars[0], 1);
            sdrgpu::tma::mbar_init(&bars[1], 1);
            sdrgpu::tma::fence_barrier_init();
        }
        __syncthreads();
        if (tid == 0) {
            issue(0);
            if (!kDecim && n_tiles > 1) issue(1);
        }
    }
    __syncthreads();

    // Software pipeline over the tiles: warps 0 .. 2 (the filter group, its own named barrier) run the half-band cascade and
    // the FIR of tile t + 1 while the first thread of warp 3 runs the serial squelch chain of tile t; then all four warps
    // demodulate tile t.  The chain (20 cycles of dependent FP64 latency per sample, 46 % of a tile's time when the CTA
    // ran its phases one after the other) now hides behind the next tile's filters; filt / pw / gate are double buffered.
    // (Spreading the CTAs' chain warps over the SM's four schedulers with a per-SM ticket was measured: no change, 2.00 ms.)
    constexpr int chain_warp = 3;
    const bool chain_thread = tid == 32 * chain_warp, filter_thread = (tid >> 5) != chain_warp;
    const int ft = tid;   // index within the filter group (warps 0 .. 2)
    auto filter_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(kNbfmFilterThreads) : "memory"); };
    auto filters = [&](int t) {
        const int Tt = tile_outputs(t);
        float2 *filt_t = filt + (t & 1) * T;
        double *pw_t = pw + (t & 1) * T;
        const int w0 = d * Tt + p.hist0;           // raw samples in this tile's window
        float2 *raw = (t & 1) ? raw1 : raw0;
        if (p.use_bulk) {
            if constexpr (kDecim) sdrgpu::tma::mbar_wait(&bars[0], (uint32_t)(t & 1));
            else sdrgpu::tma::mbar_wait(&bars[t & 1], (uint32_t)((t >> 1) & 1));
        } else {
            const long long base = (long long)t * d * T - p.hist0;
            for (int i = ft; i < w0; i += kNbfmFilterThreads) {
                const long long g = base + i;
                raw[i] = g < 0 ? hist[p.hist0 + g] : in[g];
            }
            filter_sync();
        }

        // ---- half-band cascade: z_s[i] = sum_{j even} c[j] (x[2i + j] + x[2i + L-1-j]) + x[2i + (L-1)/2] * 0.5, L = 4 P - 1.
        // A stage multiplies only even-indexed input samples: with E[k] = x[2k], O[k] = x[2k + 1] it is the symmetric FIR
        //     z[i] = sum_{t < P} c[2t] (E[i + t] + E[i + 2P - 1 - t]) + O[i + P - 1] * 0.5        (t ascending = j ascending; P even)
        // and a thread that owns four consecutive outputs slides two 6-entry register windows over E, one upwards from
        // E[i] and one downwards from E[i + 2P + 3]: two LDS.128 per two taps x four outputs (was: two LDS.64 per tap and
        // output, two-way bank conflicted).  The raw window is de-interleaved into the planes first; every stage writes the
        // planes of the next one, the last writes the FIR's input.
        int cnt = w0;
        int delta = 0;    // the FIR's input is stored shifted by delta so that its register windows start on multiples of 4
        if constexpr (kDecim) {
            auto ld2 = [](const float2 *plane, int k, float2 &a, float2 &b) {   // skewed entries k (even), k + 1
                const float4 v = *reinterpret_cast<const float4 *>(plane + nbfm_skew(k));
                a = make_float2(v.x, v.y);
                b = make_float2(v.z, v.w);
            };
            for (int k = ft; 2 * k < w0; k += kNbfmFilterThreads) {
                const float4 v = *reinterpret_cast<const float4 *>(raw + 2 * k);   // (w0 is even: hist0 and d Tt are)
                pe0[nbfm_skew(k)] = make_float2(v.x, v.y);
                po0[k] = make_float2(v.z, v.w);
            }
            filter_sync();
            // the raw window has been consumed: its buffer can take the window of tile t + 1, which arrives while this
            // tile's cascade and FIR run
            if (p.use_bulk && ft == 0 && t + 1 < n_tiles) {
                sdrgpu::tma::fence_proxy_async();
                issue(t + 1);
            }
            {   // count of the last stage's outputs -> the FIR's `off` -> delta
                int c2 = w0;
                for (int s = 0; s < S; s++) c2 = (c2 - (taps.stage[s].length - 1)) >> 1;
                delta = (7 - (c2 - Tt)) & 3;   // (off - 7 + delta) % 4 == 0
            }
            for (int s = 0; s < S; s++) {
                const HalfBandTaps &hb = taps.stage[s];
                const int L = hb.length, P = (L + 1) >> 2;
                const int n_out = (cnt - (L - 1)) >> 1;
                const float2 *E = (s & 1) ? pe1 : pe0, *O = (s & 1) ? po1 : po0;
                float2 *En = (s & 1) ? pe0 : pe1, *On = (s & 1) ? po0 : po1;
                const bool last = s == S - 1;
                for (int i0 = 4 * ft; i0 < n_out; i0 += 4 * kNbfmFilterThreads) {
                    // lo = E[i0 + t .. i0 + t + 5], hi = E[i0 + 2P - 2 - t .. i0 + 2P + 3 - t] for the tap pair (t, t + 1).
                    // i0, 2P and the main loop's t are multiples of 4, so the skewed positions are constant steps from two
                    // pointers that move 6 entries per four taps (no per-load index arithmetic).
                    float2 lo[6], hi[6];
                    const float2 *plo = E + nbfm_skew(i0), *phi = E + nbfm_skew(i0 + 2 * P - 4);
                    auto ldp = [](const float2 *q, float2 &a, float2 &b) {
                        const float4 v = *reinterpret_cast<const float4 *>(q);
                        a = make_float2(v.x, v.y);
                        b = make_float2(v.z, v.w);
                    };
                    ldp(plo, lo[0], lo[1]);
                    ldp(plo + 2, lo[2], lo[3]);
                    ldp(plo + 6, lo[4], lo[5]);
                    ldp(phi + 2, hi[0], hi[1]);
                    ldp(phi + 6, hi[2], hi[3]);
                    ldp(phi + 8, hi[4], hi[5]);
                    // I and Q rails packed, every operation separately rounded like the Java's a + b, c * sum, acc + product.  The
                    // product is an FFMA2 with a -0.0 addend (exact: x y + -0 is the rounded product, signed zeros included)
                    // whose value the compiler cannot see (a kernel parameter): ptxas contracts mul.rn.f32x2 + add.rn.f32x2
                    // -- and an FFMA2 with a literal -0.0 addend + add -- into ONE FFMA2 whatever -fmad says (checked in the
                    // SASS), which would round once where the Java rounds twice.
                    const float2 nz = make_float2(p.neg_zero, p.neg_zero);
                    float2 az[4] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
                    auto pair = [&](float h0, float h1) {
                        const float2 g0 = make_float2(h0, h0), g1 = make_float2(h1, h1);
#pragma unroll
                        for (int j = 0; j < 4; j++)   // tap t: E[i0 + j + t] = lo[j], E[i0 + j + 2P - 1 - t] = hi[j + 1]
                            az[j] = __fadd2_rn(az[j], __ffma2_rn(g0, __fadd2_rn(lo[j], hi[j + 1]), nz));
#pragma unroll
                        for (int j = 0; j < 4; j++)   // tap t + 1: lo[j + 1], hi[j]
                            az[j] = __fadd2_rn(az[j], __ffma2_rn(g1, __fadd2_rn(lo[j + 1], hi[j]), nz));
                    };
                    auto slide = [&](const float2 *ql, const float2 *qh) {   // windows of the next tap pair
#pragma unroll
                        for (int m = 0; m < 4; m++) lo[m] = lo[m + 2];
                        ldp(ql, lo[4], lo[5]);
#pragma unroll
                        for (int m = 5; m >= 2; m--) hi[m] = hi[m - 2];
                        ldp(qh, hi[0], hi[1]);
                    };
                    int t2 = 0;
                    for (; t2 + 3 < P; t2 += 4) {
                        pair(hb.c[2 * t2], hb.c[2 * t2 + 2]);
                        slide(plo + 8, phi);                       // E[i0 + t2 + 6 ..], E[i0 + 2P - 4 - t2 ..]
                        pair(hb.c[2 * t2 + 4], hb.c[2 * t2 + 6]);
                        if (t2 + 4 < P) slide(plo + 12, phi - 4);  // E[i0 + t2 + 8 ..], E[i0 + 2P - 6 - t2 ..]
                        plo += 6;
                        phi -= 6;
                    }
                    if (P & 2) pair(hb.c[2 * t2], hb.c[2 * t2 + 2]);   // P = 6 (23 taps): a last pair on the windows just loaded
                    const float ai[4] = {az[0].x, az[1].x, az[2].x, az[3].x}, aq[4] = {az[0].y, az[1].y, az[2].y, az[3].y};
                    float2 z[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const float2 mid = O[i0 + j + P - 1];
                        z[j] = make_float2(__fadd_rn(ai[j], __fmul_rn(mid.x, 0.5f)), __fadd_rn(aq[j], __fmul_rn(mid.y, 0.5f)));
                    }
                    // (outputs at or behind n_out are computed from stale entries and land in slack nobody reads)
                    if (last) {
#pragma unroll
                        for (int j = 0; j < 4; j++) zs[nbfm_skew(i0 + j + delta)] = z[j];
                    } else {
                        *reinterpret_cast<float4 *>(En + nbfm_skew(i0 >> 1)) = make_float4(z[0].x, z[0].y, z[2].x, z[2].y);
                        *reinterpret_cast<float4 *>(On + (i0 >> 1)) = make_float4(z[1].x, z[1].y, z[3].x, z[3].y);
                    }
                }
                filter_sync();
                cnt = n_out;
            }
        }

        // ---- FIR: y[i] = fma chain over k of z[i + off - k] h[k] (k ascending), * gain; then the squelch's alpha * power.
        // Four outputs per thread on an 11-sample register window: 8 taps = 32 FFMA2 (I and Q rails packed) per 8 samples
        // loaded (decimating variant: four LDS.128 from the skewed buffer; else eight LDS.64 from the raw window).
        const int off = cnt - Tt;                 // newest sample of output i is z[i + off]; off >= KP - 1 (hist0)
        for (int i0 = 4 * ft; i0 < Tt; i0 += 4 * kNbfmFilterThreads) {
            float2 acc[4];
            auto zat = [&](int i) { return kDecim ? zs[nbfm_skew(i + delta)] : raw[i]; };
#pragma unroll
            for (int j = 0; j < 4; j++) acc[j] = N > 0 ? make_float2(0.0f, 0.0f) : zat(min(i0 + j, Tt - 1) + off);
            if (N > 0) {
                // w[m] = z[i0 + off - (KP - 1) + m]: output j, tap k reads w[j + KP - 1 - k]; x[] = w[base .. base + 10]
                const int w_at = i0 + off - (KP - 1);               // index of w[0]
                const int top = cnt - 1 - w_at;                     // highest valid index of w (a partial group at the tile end)
                float2 x[12];
                int base = KP - 8;
                // decimating variant: w_at + base + delta = i0 + off - 7 + delta - k is a multiple of 4 (delta), so the skewed
                // positions of a window are constant steps from one pointer that moves 12 entries per 8 taps; entries past
                // `top` are stale but in bounds and only reach outputs that are not stored
                const float2 *px = zs + nbfm_skew(kDecim ? w_at + base + delta : 0);
                if constexpr (kDecim) {
                    constexpr int at[6] = {0, 2, 6, 8, 12, 14};   // nbfm_skew(0, 2, .., 10)
#pragma unroll
                    for (int m = 0; m < 12; m += 2) {
                        const float4 v = *reinterpret_cast<const float4 *>(px + at[m >> 1]);
                        x[m] = make_float2(v.x, v.y);
                        x[m + 1] = make_float2(v.z, v.w);
                    }
                } else {
#pragma unroll
                    for (int m = 0; m < 11; m++) x[m] = raw[w_at + min(base + m, top)];
                }
                for (int k = 0; k < KP; k += 8) {
                    const float4 ha = *reinterpret_cast<const float4 *>(hs + k), hb = *reinterpret_cast<const float4 *>(hs + k + 4);
                    const float h8[8] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const float2 hh = make_float2(h8[u], h8[u]);
#pragma unroll
                        for (int j = 0; j < 4; j++) acc[j] = __ffma2_rn(x[j + 7 - u], hh, acc[j]);
                    }
                    if (k + 8 < KP) {
                        base -= 8;
                        x[8] = x[0];
                        x[9] = x[1];
                        x[10] = x[2];
                        if constexpr (kDecim) {
                            constexpr int at[4] = {0, 2, 6, 8};
                            px -= 12;
#pragma unroll
                            for (int m = 0; m < 8; m += 2) {
                                const float4 v = *reinterpret_cast<const float4 *>(px + at[m >> 1]);
                                x[m] = make_float2(v.x, v.y);
                                x[m + 1] = make_float2(v.z, v.w);
                            }
                        } else {
#pragma unroll
                            for (int m = 0; m < 8; m++) x[m] = raw[w_at + base + m];
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; j++) acc[j] = make_float2(__fmul_rn(acc[j].x, p.fir_gain), __fmul_rn(acc[j].y, p.fir_gain));
            }
            // PowerSquelch.process(double, double): inphase * inphase + quadrature * quadrature, then alpha * power
            double pwr[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const double di = (double)acc[j].x, dq = (double)acc[j].y;
                pwr[j] = __dmul_rn(p.alpha, __dadd_rn(__dmul_rn(di, di), __dmul_rn(dq, dq)));
            }
            if (i0 + 4 <= Tt) {   // (T is a multiple of 4 and the halves are 16-byte aligned: two 16-byte stores each)
                *reinterpret_cast<float4 *>(filt_t + i0) = make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y);
                *reinterpret_cast<float4 *>(filt_t + i0 + 2) = make_float4(acc[2].x, acc[2].y, acc[3].x, acc[3].y);
                *reinterpret_cast<double2 *>(pw_t + i0) = make_double2(pwr[0], pwr[1]);
                *reinterpret_cast<double2 *>(pw_t + i0 + 2) = make_double2(pwr[2], pwr[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    if (i0 + j < Tt) {
                        filt_t[i0 + j] = acc[j];
                        pw_t[i0 + j] = pwr[j];
                    }
                }
            }
        }
        filter_sync();
        if (!kDecim && p.use_bulk && ft == 0 && t + 2 < n_tiles) {
            sdrgpu::tma::fence_proxy_async();
            issue(t + 2);
        }

    };
    auto squelch_chain = [&](int t) {
        const int Tt = tile_outputs(t);
        const float2 *filt_t = filt + (t & 1) * T;
        const double *pw_t = pw + (t & 1) * T;
        uint32_t *gate_t = gate + (t & 1) * gate_words;
        // ---- power squelch: the serial part.  The IIR is a two-operation dependent chain per sample; its comparisons are
        // collected 32 at a time, and the ramp state machine runs on those words -- while the state is stable (open, or
        // shut) a word is one test -- so that the one thread issues ~5 instructions per sample, not one per state test.
        {
            int last_gated = -1;     // -1: the sample carried in s_prev
            if (p.squelch) {
                const double one_minus = 1.0 - p.alpha, threshold = s_threshold;
                double output = st.output;
                int state = st.state, ramp_count = st.ramp_count;
                const int ramp = p.ramp;
                for (int k0 = 0; k0 < Tt; k0 += 32) {
                    const int n = min(32, Tt - k0);
                    uint32_t mute_bits = 0;
                    if (n == 32) {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            const double2 pp = *reinterpret_cast<const double2 *>(pw_t + k0 + j);
                            output = __dadd_rn(__dmul_rn(output, one_minus), pp.x);
                            mute_bits |= (output < threshold ? 1u : 0u) << j;
                            output = __dadd_rn(__dmul_rn(output, one_minus), pp.y);
                            mute_bits |= (output < threshold ? 1u : 0u) << (j + 1);
                        }
                    } else {
                        for (int j = 0; j < n; j++) {
                            output = __dadd_rn(__dmul_rn(output, one_minus), pw_t[k0 + j]);
                            mute_bits |= (output < threshold ? 1u : 0u) << j;
                        }
                    }
                    const uint32_t all = n == 32 ? 0xffffffffu : ((1u << n) - 1u);
                    // kStatus: bit j = output k0 + j ends an assembler buffer (tiles and buffers need not line up).
                    // Within the ramp machine the state changes exactly where the gate flips (ATTACK / MUTE -> UNMUTE,
                    // DECAY / UNMUTE -> MUTE), so a buffer's CHANGED bit is "an edge of the gate in it"; the gate in
                    // front of a word is that of the state it starts from.
                    uint32_t end_bits = 0;
                    if constexpr (kStatus) {
                        const int g0 = t * T + k0;
                        for (; buffer_end < g0 + n; buffer_end += p.buffer_out) end_bits |= 1u << (buffer_end - g0);
                    }
                    auto report = [&](bool edge) {
                        *status_at++ = (uint8_t)(state | (changed || edge ? SDRGPU_SQUELCH_CHANGED : 0));
                        changed = false;
                    };
                    uint32_t on_bits;
                    if (state == 3 && mute_bits == 0) {
                        on_bits = all;            // UNMUTE and never below the threshold: every sample demodulated
                        if constexpr (kStatus)    // (no edge in a stable word)
                            for (uint32_t e = end_bits; e; e &= e - 1) report(false);
                    } else if (state == 2 && mute_bits == all) {
                        on_bits = 0;              // MUTE and never above it
                        if constexpr (kStatus)
                            for (uint32_t e = end_bits; e; e &= e - 1) report(false);
                    } else {
                        on_bits = 0;
                        const uint32_t gate_in = (uint32_t)state & 1u;   // UNMUTE / DECAY: the gate is on
                        uint32_t open = 0xffffffffu;                     // bits of this word in the current buffer
                        for (int j = 0; j < n; j++) {
                            if (squelch_step(state, ramp_count, (mute_bits >> j) & 1u, ramp)) on_bits |= 1u << j;
                            if constexpr (kStatus) {
                                if ((end_bits >> j) & 1u) {
                                    const uint32_t upto = 0xffffffffu >> (31 - j);
                                    report(((on_bits ^ ((on_bits << 1) | gate_in)) & upto & open) != 0);
                                    open = ~upto;
                                }
                            }
                        }
                        if constexpr (kStatus) changed |= ((on_bits ^ ((on_bits << 1) | gate_in)) & all & open) != 0;
                    }
                    gate_t[k0 >> 5] = on_bits;
                    if (on_bits) last_gated = k0 + 31 - __clz(on_bits);
                }
                st.output = output;
                st.state = state;
                st.ramp_count = ramp_count;
            } else {
                last_gated = Tt - 1;
            }
            // the demodulator's previous sample after this tile (written after the FM pass below has read the old one)
            st.prev_i = last_gated >= 0 ? filt_t[last_gated].x : s_prev[0];
            st.prev_q = last_gated >= 0 ? filt_t[last_gated].y : s_prev[1];
        }
    };
    auto fm_pass = [&](int t) {
        const int Tt = tile_outputs(t);
        const float2 *filt_t = filt + (t & 1) * T;
        const uint32_t *gate_t = gate + (t & 1) * gate_words;
        // ---- FM discriminator epilogue
        if (p.out) {
            float *y = p.out + (size_t)c * p.out_stride + (size_t)t * T;
            const float pi0 = s_prev[0], pq0 = s_prev[1];
            for (int k = tid; k < Tt; k += kNbfmThreads) {
                float v = 0.0f;
                if (!p.squelch || ((gate_t[k >> 5] >> (k & 31)) & 1u)) {
                    // demodulated against the most recent demodulated sample (the demodulator's state does not move while muted)
                    int q = k - 1;
                    if (p.squelch) {
                        int wd = k >> 5;
                        uint32_t below = gate_t[wd] & ((1u << (k & 31)) - 1u);
                        while (below == 0 && wd > 0) below = gate_t[--wd];
                        q = below ? 32 * wd + 31 - __clz(below) : -1;
                    }
                    const float pi_ = q >= 0 ? filt_t[q].x : pi0, pq = q >= 0 ? filt_t[q].y : pq0;
                    v = fm_angle(filt_t[k].x, filt_t[k].y, pi_, pq, p.fm_gain);
                }
                y[k] = v;
            }
        }
    };

    if (filter_thread) filters(0);
    __syncthreads();
    for (int t = 0; t < n_tiles; t++) {
        if (chain_thread) {
            if (t > 0) {   // FMDemodulator.mPreviousI / Q after tile t - 1 (its FM pass has read the old values)
                s_prev[0] = st.prev_i;
                s_prev[1] = st.prev_q;
            }
            squelch_chain(t);
        } else if (filter_thread && t + 1 < n_tiles) {
            filters(t + 1);
        }
        __syncthreads();
        fm_pass(t);
        __syncthreads();
    }

    // history of the next call: the last hist0 samples of [hist | in]
    if (p.hist_out) {
        float2 *ho = p.hist_out + (size_t)c * p.hist_out_stride;
        for (int i = tid; i < p.hist0; i += kNbfmThreads) {
            const long long g = (long long)p.n_new - p.hist0 + i;
            ho[i] = g < 0 ? hist[p.hist0 + g] : in[g];
        }
    }
    if (chain_thread) p.sq[c] = st;
}

sdrgpu_status nbfm_fused_launch(const FmLaunch &a)
{
    NbfmHistory &h = *a.fused;
    NbfmParams q{};
    q.hist = h.d[h.cur];
    q.hist_stride = h.hist0;
    q.in = a.in;
    q.in_stride = a.in_stride;
    q.hist_out = h.d[h.cur ^ 1];
    q.hist_out_stride = h.hist0;
    q.n_new = a.n;
    q.hist0 = h.hist0;
    q.n_stages = a.n_stages;
    q.n_fir = a.n_fir;
    q.fir_gain = a.fir_gain;
    const int d = 1 << a.n_stages;
    static const int tile_env = getenv("SDRGPU_NBFM_TILE") ? atoi(getenv("SDRGPU_NBFM_TILE")) : 256;
    int tile = tile_env >= 4 ? (tile_env & ~3) : 256;
    while (d * tile < h.hist0) tile *= 2;   // a window starts at most one tile back
    q.tile_out = tile;
    q.window_cap = (d * tile + h.hist0 + 1) & ~1;
    q.use_bulk = (reinterpret_cast<uintptr_t>(q.in) % 16 == 0) && (q.in_stride % 2 == 0) && (a.n_stages > 0 || a.n % 2 == 0);
    q.squelch = a.squelch;
    q.alpha = a.alpha;
    q.thresholds = a.thresholds;
    q.ramp = a.ramp;
    q.fm_gain = a.gain;
    q.sq = a.states;
    q.out = a.out;
    q.out_stride = a.out_stride;
    q.status = a.squelch ? a.status : nullptr;
    q.status_stride = a.status_stride;
    q.buffer_out = a.buffer_out;
    q.n_channels = a.n_channels;
    q.neg_zero = -0.0f;
    NbfmStageTaps st{};
    for (int i = 0; i < a.n_stages; i++) st.stage[i] = a.stages[i];
    const int first_cnt = a.n_stages >= 1 ? ((d * tile + h.hist0 - (a.stages[0].length - 1)) >> 1) : 0;
    nbfm_fused_layout(q, first_cnt);
    const size_t smem = nbfm_fused_smem(q);
    static bool attr_set = false;
    if (!attr_set) {
        SDRGPU_CUDA(cudaFuncSetAttribute(nbfm_fused_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        SDRGPU_CUDA(cudaFuncSetAttribute(nbfm_fused_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        SDRGPU_CUDA(cudaFuncSetAttribute(nbfm_fused_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        SDRGPU_CUDA(cudaFuncSetAttribute(nbfm_fused_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        attr_set = true;
    }
    auto *kernel = a.n_stages >= 1 ? (q.status ? nbfm_fused_kernel<true, true> : nbfm_fused_kernel<true, false>)
                                   : (q.status ? nbfm_fused_kernel<false, true> : nbfm_fused_kernel<false, false>);
    kernel<<<a.n_channels, kNbfmThreads, smem, a.stream>>>(q, st, *a.fir);
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    h.cur ^= 1;
    return SDRGPU_OK;
}

}  // namespace

namespace sdrgpu {

bool nbfm_fused_fits(const sdrgpu_bank_config &cfg, const HalfBandTaps *stages, int n_stages, int n_fir, int *hist0)
{
    if (!is_fm(cfg.demod) || cfg.agc || n_stages > kMaxFusedStages) return false;
    for (int i = 0; i < n_stages; i++)   // the kernel's plane formulation of a half-band stage: L = 4 P - 1 with P even (15 / 23 / 63 are)
        if (stages[i].length % 8 != 7) return false;
    // raw history a tile's first output needs: N - 1 samples of the last stage, each stage back doubling them and adding
    // its own L - 1 (the filters are pure functions of the stream, so the samples are recomputed, not carried)
    int lo = n_fir > 0 ? fir_padded_taps(n_fir) - 1 : 0;   // the FIR reads whole groups of 8 (zero-padded) taps
    for (int i = n_stages - 1; i >= 0; i--) lo = 2 * lo + (stages[i].length - 1);
    *hist0 = (lo + 1) & ~1;
    return true;
}

sdrgpu_status fm_create(int n_channels, double threshold, SquelchState **d_states, double **d_thresholds)
{
    std::vector<SquelchState> init((size_t)n_channels);
    std::memset(init.data(), 0, sizeof(SquelchState) * (size_t)n_channels);
    for (auto &s : init) s.state = 2;  // PowerSquelch starts MUTE (PowerSquelch.java:18)
    SDRGPU_CUDA(cudaMalloc(d_states, sizeof(SquelchState) * (size_t)n_channels));
    SDRGPU_CUDA(cudaMemcpy(*d_states, init.data(), sizeof(SquelchState) * (size_t)n_channels, cudaMemcpyHostToDevice));
    const std::vector<double> thresholds((size_t)n_channels, threshold);
    SDRGPU_CUDA(cudaMalloc(d_thresholds, sizeof(double) * (size_t)n_channels));
    SDRGPU_CUDA(cudaMemcpy(*d_thresholds, thresholds.data(), sizeof(double) * (size_t)n_channels, cudaMemcpyHostToDevice));
    return SDRGPU_OK;
}

sdrgpu_status fm_set_threshold(double *d_thresholds, int n_channels, int channel, double threshold, cudaStream_t stream)
{
    const int first = channel < 0 ? 0 : channel, count = channel < 0 ? n_channels : 1;
    set_threshold_kernel<<<(count + 255) / 256, 256, 0, stream>>>(d_thresholds + first, count, threshold);
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    return SDRGPU_OK;
}

sdrgpu_status fm_launch(const FmLaunch &a)
{
    if (a.fused) return nbfm_fused_launch(a);
    const int C = a.n_channels;
    cudaStream_t s = a.stream;
    const uint8_t *gate = nullptr;
    if (a.squelch) {
        squelch_gate_kernel<<<(C + 63) / 64, 64, 0, s>>>(a.in, a.in_stride, a.n, a.states, a.gate, a.in_stride, a.alpha,
                                                         a.thresholds, a.ramp, a.status, a.status_stride, a.buffer_out, C);
        count_launch();
        SDRGPU_CUDA(cudaGetLastError());
        gate = a.gate;
    }
    if (a.out) {
        dim3 grid((a.n + 255) / 256 > 64 ? 64 : (a.n + 255) / 256, C);
        fm_kernel<<<grid, 256, 0, s>>>(a.in, a.in_stride, a.n, gate, a.in_stride, a.states, a.gain, a.out, a.out_stride);
        count_launch();
        SDRGPU_CUDA(cudaGetLastError());
    }
    fm_carry_kernel<<<(C + 63) / 64, 64, 0, s>>>(a.in, a.in_stride, a.n, gate, a.in_stride, a.states, C);
    count_launch();
    SDRGPU_CUDA(cudaGetLastError());
    return SDRGPU_OK;
}

}  // namespace sdrgpu
