// The channelizer's output stage for "special" channels: two-bin channels (post_channel_kernel) and one-bin channels with
// a frequency offset (osc_produce_kernel + osc_mix_kernel, or pfb2_kernel mixing the oscillators in where it stores).
// The filter bank leaves their rows at gain 1 (bin values after the 1/M of the inverse FFT); this stage finishes them in
// place on the channelizer's stream.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "outputs.cuh"

using namespace sdrgpu;

namespace {

// Oscillator.rotate + Complex.fastNormalize (J/dsp/mixer/Oscillator.java:42-68): current *= angle, then rescaled by
// 1.9999 - |current|^2
__device__ __forceinline__ float2 osc_rotate(float2 cur, float2 angle)
{
    const float2 n = mix_complex(cur, angle);
    const float norm = __fadd_rn(__fmul_rn(n.x, n.x), __fmul_rn(n.y, n.y));
    const float scalor = __fsub_rn(1.9999f, norm);
    return make_float2(__fmul_rn(n.x, scalor), __fmul_rn(n.y, scalor));
}

// ---------------------------------------------------------------------------------------------------------------
// Post-processing of the two-bin channels, in place on their rows, one warp per channel:
//   two-bin channels  TwoChannelOutputProcessor.process + TwoChannelSynthesizerM2.process + FS4DownConverter
//                     (J/dsp/filter/channelizer/output/TwoChannelOutputProcessor.java:98-121,
//                      J/dsp/filter/channelizer/TwoChannelSynthesizerM2.java:90-158, J/dsp/mixer/FS4DownConverter.java:32-68)
//   frequency offset  Oscillator mix (J/dsp/mixer/Oscillator.java:42-68, AbstractOscillator.java:102-116): the rotator
//                     is a float recursion with fastNormalize, so it runs as a sequential chain that every lane
//                     walks, lane i keeping the value of sample i
//   gain              ReusableComplexBuffer.applyGain: samples[x] = (float)(samples[x] * (double) gain)
// ---------------------------------------------------------------------------------------------------------------
template <bool ROUTED>
__global__ void __launch_bounds__(32) post_channel_kernel(float *out, long long out_stride, const float *out2,
                                                          long long out2_stride, int n, const PostChannel *chans,
                                                          PostState *states, const __grid_constant__ SynthFilter filt,
                                                          float *const *rows, long long col)
{
    __shared__ float4 ent[kMaxSynthEntries + 32];
    const int lane = threadIdx.x;
    const PostChannel c = chans[blockIdx.x];
    PostState *st = states + blockIdx.x;
    float2 *row = reinterpret_cast<float2 *>(channel_row<ROUTED>(out, out_stride, rows, col, c.row));
    const float2 *row2 = c.row2 >= 0 ? reinterpret_cast<const float2 *>(out2 + (size_t)c.row2 * out2_stride) : nullptr;
    const int H = filt.entries - 1;   // history entries a sample needs besides its own
    const float2 angle = make_float2(c.angle_i, c.angle_q);
    float2 cur = make_float2(st->cur_i, st->cur_q);
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
            // AbstractOscillator.mixComplex: sample * current, then rotate()
            float2 mine = cur;
            const int count = min(32, n - base);
            for (int i = 0; i < count; i++) {
                if (i == lane) mine = cur;
                cur = osc_rotate(cur, angle);
            }
            v = mix_complex(v, mine);
        }
        v.x = __double2float_rn(__dmul_rn((double)v.x, c.gain));
        v.y = __double2float_rn(__dmul_rn((double)v.y, c.gain));
        if (valid) row[k] = v;
    }
    if (lane == 0) {
        st->cur_i = cur.x;
        st->cur_q = cur.y;
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
// The `count` oscillator values from `cur` on into ring slots pos, pos + 1, ... (wrapping at ring_len); leaves cur at the
// value after them
__device__ __forceinline__ void osc_fill(float2 *r, int ring_len, int pos, int count, float2 &cur, float2 angle)
{
    int k = 0;
    while (k < count) {
        if ((pos & 1) == 0 && k + 8 <= count && pos + 8 <= ring_len) {
            // eight steps with nothing but the recursion between them, then four 16-byte stores (ring_len is even and
            // the rows are 16-byte aligned)
            float4 w[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                w[j].x = cur.x;
                w[j].y = cur.y;
                cur = osc_rotate(cur, angle);
                w[j].z = cur.x;
                w[j].w = cur.y;
                cur = osc_rotate(cur, angle);
            }
#pragma unroll
            for (int j = 0; j < 4; j++) reinterpret_cast<float4 *>(r + pos)[j] = w[j];
            pos += 8;
            k += 8;
        } else {
            r[pos] = cur;
            cur = osc_rotate(cur, angle);
            pos += 1;
            k += 1;
        }
        if (pos >= ring_len) pos = 0;
    }
}

__global__ void __launch_bounds__(32) osc_produce_kernel(const MixChannel *__restrict__ chans, float2 *__restrict__ state,
                                                           float2 *__restrict__ ring, int ring_len, long long start, int count,
                                                           int n_mix)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_mix) return;
    const float2 angle = make_float2(chans[ch].angle_i, chans[ch].angle_q);
    float2 cur = state[ch];
    float2 *r = ring + (size_t)ch * ring_len;
    const int pos = (int)(start % ring_len);
    osc_fill(r, ring_len, pos, count, cur, angle);
    state[ch] = cur;
}

// ---------------------------------------------------------------------------------------------------------------
// A new frequency offset for running one-bin channels (ChannelOutputProcessor.setFrequencyOffset -> Oscillator.update:
// only the angle changes).  The rings hold the values of blocks start .. start + count - 1 (slot k % ring_len: the phasor
// that multiplies block k), produced with the old angle.  Slot `start` stays: the next block is mixed with the phasor the
// old angle produced.  Slots start + 1 .. start + count - 1 and the producer's state are rewritten from it with the new
// angle, one thread per changed channel, with the producer's arithmetic.  A channel that starts mixing (held_row >= 0)
// starts from the phasor it held, which also goes into slot `start`.  Calls still in flight read slots below `start`
// only, and ring_len = 2 max_blocks + 9 > count, so no slot they read is rewritten.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) osc_reproduce_kernel(MixChannel *__restrict__ chans, float2 *__restrict__ state,
                                                             float2 *__restrict__ ring, int ring_len, long long start, int count,
                                                             const float2 *__restrict__ held,
                                                             const __grid_constant__ OffsetChanges changes)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= changes.n) return;
    const OffsetChange c = changes.c[i];
    const float2 angle = make_float2(c.angle_i, c.angle_q);
    // the producer's angle from here on (it runs on this kernel's stream)
    chans[c.index].angle_i = c.angle_i;
    chans[c.index].angle_q = c.angle_q;
    float2 *r = ring + (size_t)c.index * ring_len;
    const int pos = (int)(start % ring_len);
    float2 cur = c.held_row >= 0 ? held[c.held_row] : (count > 0 ? r[pos] : state[c.index]);
    if (count > 0) {
        if (c.held_row >= 0) r[pos] = cur;
        cur = osc_rotate(cur, angle);
        osc_fill(r, ring_len, pos + 1 == ring_len ? 0 : pos + 1, count - 1, cur, angle);
    }
    state[c.index] = cur;
}

// two-bin channels: the synthesizer's Oscillator takes the new angle, on the channelizer's stream
__global__ void post_angle_kernel(PostChannel *chans, const __grid_constant__ OffsetChanges changes)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= changes.n) return;
    chans[changes.c[i].index].angle_i = changes.c[i].angle_i;
    chans[changes.c[i].index].angle_q = changes.c[i].angle_q;
}

// The mix set changes (outputs_update): one block per old mix channel m.  A kept channel that keeps mixing moves its live
// ring window (blocks start .. start + count - 1) and producer state to its new row to[m].x; one that stops mixing
// (to[m].x < 0) holds, at its new selection index to[m].y, the phasor its next block would have used; a removed one
// (both -1) is dropped.
__global__ void osc_carry_kernel(const float2 *old_state, const float2 *old_ring, const int2 *to, float2 *state,
                                 float2 *ring, float2 *held, int ring_len, long long start, int count)
{
    const int m = blockIdx.x, d = to[m].x;
    const float2 *src = old_ring + (size_t)m * ring_len;
    if (d < 0) {
        if (threadIdx.x == 0 && to[m].y >= 0) held[to[m].y] = count > 0 ? src[start % ring_len] : old_state[m];
        return;
    }
    for (int k = threadIdx.x; k < count; k += blockDim.x) {
        const int pos = (int)((start + k) % ring_len);
        ring[(size_t)d * ring_len + pos] = src[pos];
    }
    if (threadIdx.x == 0) state[d] = old_state[m];
}

// A table indexed by row follows a selection edit: entry i of the new table is entry from[i] of the old one, or `init`
// for a new channel (from[i] < 0).  Two-bin channels' PostState (phasor, top_block, fs4, synthesizer history) and the
// phasors d_held keeps per selected channel.
template <class T>
__global__ void gather_kernel(const T *src, const int *from, T *dst, int n, const __grid_constant__ T init)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = from[i] >= 0 ? src[from[i]] : init;
}

// grid (ceil(n / 256), n_mix): row[k] = (float)((double)(row[k] * osc[start + k]) * gain)
template <bool ROUTED>
__global__ void osc_mix_kernel(float *out, long long out_stride, const MixChannel *__restrict__ chans,
                               const float2 *__restrict__ ring, int ring_len, long long start, int n, float *const *rows,
                               long long col)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const MixChannel c = chans[blockIdx.y];
    float2 *row = reinterpret_cast<float2 *>(channel_row<ROUTED>(out, out_stride, rows, col, c.row));
    const float2 m = mix_complex(row[k], ring[(size_t)blockIdx.y * ring_len + (int)((start + k) % ring_len)]);
    row[k] = make_float2(__double2float_rn(__dmul_rn((double)m.x, c.gain)), __double2float_rn(__dmul_rn((double)m.y, c.gain)));
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------

// osc_produce_kernel: the next `count` values of every ring on `stream`
void produce(ChanOutputs &o, int count, cudaStream_t stream)
{
    osc_produce_kernel<<<(o.n_mix + 31) / 32, 32, 0, stream>>>(o.d_mix, o.d_mix_state, o.d_osc, o.osc_ring_len,
                                                               o.osc_produced, count, o.n_mix);
    count_launch();
    o.osc_produced += count;
}

// The values of the next calls, on the side stream behind the last kernel that read the rings (their slots' last reader).
// The producer is an ordinary small kernel there: it shares the SMs with whatever runs beside it, and its cost is measured
// as such (bench.py: with_frequency_corrected_channels; DESIGN.md section 4 has the history).
sdrgpu_status produce_ahead(ChanOutputs &o, int count)
{
    if (o.mix_recorded) SDRGPU_CUDA(cudaStreamWaitEvent(o.osc_stream, o.ev_mix, 0));
    produce(o, count, o.osc_stream);
    SDRGPU_CUDA(cudaGetLastError());
    SDRGPU_CUDA(cudaEventRecord(o.ev_osc, o.osc_stream));
    o.osc_pending = true;
    return SDRGPU_OK;
}

// The rings hold the n_blocks values from osc_consumed on, in `stream`'s order.
sdrgpu_status ensure_osc(ChanOutputs &o, int n_blocks, cudaStream_t stream)
{
    const long long have = o.osc_produced - o.osc_consumed;
    // wait for the top-up in flight only if this call reaches into what it writes (or has to produce itself)
    if (o.osc_pending && (o.osc_consumed + n_blocks > o.osc_safe || have < n_blocks)) {
        SDRGPU_CUDA(cudaStreamWaitEvent(stream, o.ev_osc, 0));
        o.osc_pending = false;
        o.osc_safe = o.osc_produced;
    }
    if (have < n_blocks) {  // first call, or a call longer than the look-ahead: produce the rest in line
        produce(o, (int)(n_blocks - have), stream);
        o.osc_safe = o.osc_produced;
    }
    return SDRGPU_OK;
}

template <class T>
void release(T *&d)
{
    cudaFree(d);
    d = nullptr;
}

void release_tables(ChanOutputs &o)
{
    release(o.d_post);
    release(o.d_post_state);
    release(o.d_out2);
    release(o.d_mix);
    release(o.d_mix_state);
    release(o.d_osc);
    release(o.d_held);
}

// the stage's buffers, once the producer is done with them; the rings restart empty
cudaError_t free_buffers(ChanOutputs &o)
{
    const cudaError_t e = o.osc_stream ? cudaStreamSynchronize(o.osc_stream) : cudaSuccess;
    release_tables(o);
    o.osc_produced = o.osc_consumed = o.osc_safe = 0;
    o.osc_pending = false;
    return e;
}

template <class T>
sdrgpu_status upload(T **d, const std::vector<T> &v)
{
    SDRGPU_CUDA(cudaMalloc(d, sizeof(T) * v.size()));
    SDRGPU_CUDA(cudaMemcpy(*d, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
    return SDRGPU_OK;
}

// Oscillator.update: anglePerSample = (float)(2 pi f / fs) at the channel rate; Complex.fromAngle(float) -> (float)cos, (float)sin
void osc_angle(long long offset_hz, int M, double sample_rate, float *angle_i, float *angle_q)
{
    const double channel_rate = 2.0 * sample_rate / (double)M;
    const float angle = (float)(2.0 * 3.14159265358979323846 * (double)offset_hz / channel_rate);
    *angle_i = (float)cos((double)angle);
    *angle_q = (float)sin((double)angle);
}

// The stage's tables for a selection: the filter bank's rows, the two-bin (post) and one-bin + offset (mix) channels, and
// each selected channel's row in those tables (post_of / mix_of, -1: none)
void plan_outputs(const std::vector<sdrgpu_output_channel> &channels, int M, double sample_rate, OutputRows *rows,
                  std::vector<PostChannel> *post, std::vector<MixChannel> *mix, std::vector<int> *post_of,
                  std::vector<int> *mix_of, int *n_two)
{
    const int n = (int)channels.size();
    std::vector<int> &sel = rows->sel;
    std::vector<double> &gd = rows->gain;
    sel.clear();
    gd.clear();
    post->clear();
    mix->clear();
    post_of->assign(n, -1);
    mix_of->assign(n, -1);
    *n_two = 0;
    for (int i = 0; i < n; i++) {
        const sdrgpu_output_channel &c = channels[i];
        const bool special = c.bin2 >= 0 || c.frequency_offset_hz != 0;
        sel.push_back(c.bin1);
        // special rows leave the filter bank at gain 1; this stage applies the gain after mixing
        gd.push_back(special ? 1.0 : c.gain);
        if (special) {
            PostChannel pc{};
            pc.row = i;
            pc.row2 = c.bin2 >= 0 ? (*n_two)++ : -1;
            // TwoChannelOutputProcessor mixes unconditionally, OneChannelOutputProcessor only with an offset
            pc.mix = 1;
            osc_angle(c.frequency_offset_hz, M, sample_rate, &pc.angle_i, &pc.angle_q);
            pc.gain = c.gain;
            if (c.bin2 >= 0) {   // two-bin: post_channel_kernel
                (*post_of)[i] = (int)post->size();
                post->push_back(pc);
            } else {             // one bin + offset: look-ahead
                (*mix_of)[i] = (int)mix->size();
                mix->push_back(MixChannel{pc.row, pc.angle_i, pc.angle_q, pc.gain});
            }
        }
    }
    for (int i = 0; i < n; i++)
        if (channels[i].bin2 >= 0) {   // scratch rows: the second bins, gain 1
            sel.push_back(channels[i].bin2);
            gd.push_back(1.0);
        }
    rows->mix_identity = (int)mix->size() == n && n == M && (int)sel.size() == n;
    for (size_t m = 0; m < mix->size() && rows->mix_identity; m++) {
        const MixChannel &x = (*mix)[m];
        if (x.row != (int)m || sel[m] != (int)m || x.gain != (*mix)[0].gain || (double)(float)x.gain != x.gain)
            rows->mix_identity = false;
    }
    rows->mix_gain = mix->empty() ? 0.0f : (float)(*mix)[0].gain;
}

sdrgpu_status ensure_osc_stream(ChanOutputs &o)
{
    if (o.osc_stream) return SDRGPU_OK;
    SDRGPU_CUDA(cudaStreamCreateWithFlags(&o.osc_stream, cudaStreamNonBlocking));
    SDRGPU_CUDA(cudaEventCreateWithFlags(&o.ev_mix, cudaEventDisableTiming));
    SDRGPU_CUDA(cudaEventCreateWithFlags(&o.ev_osc, cudaEventDisableTiming));
    return SDRGPU_OK;
}

// the OffsetChanges launches of a change list, kMaxOffsetChanges at a time
template <class Launch>
sdrgpu_status launch_changes(const std::vector<OffsetChange> &list, Launch launch)
{
    for (size_t first = 0; first < list.size(); first += kMaxOffsetChanges) {
        OffsetChanges c;
        c.n = (int)std::min(list.size() - first, (size_t)kMaxOffsetChanges);
        std::memcpy(c.c, list.data() + first, sizeof(OffsetChange) * (size_t)c.n);
        launch(c);
        count_launch();
        SDRGPU_CUDA(cudaGetLastError());
    }
    return SDRGPU_OK;
}

// TwoChannelOutputProcessor's state at creation
PostState post_init()
{
    PostState st;
    std::memset(&st, 0, sizeof(st));
    st.cur_i = 0.0f;   // Oscillator.java:24: mCurrentAngle = new Complex(0.0f, -1.0f)
    st.cur_q = -1.0f;
    st.top_block = 1;  // TwoChannelSynthesizerM2: mTopBlockIndicator = true
    return st;
}

// New angles for mix rows (a held_row starts the row from that held phasor): the look-ahead from osc_consumed on is
// rewritten on the side stream, behind the producer in flight and the last kernel that read the rings; the next call
// waits for it (osc_safe below osc_consumed + its blocks)
sdrgpu_status reproduce(ChanOutputs &o, const std::vector<OffsetChange> &list)
{
    if (list.empty()) return SDRGPU_OK;
    if (o.mix_recorded) SDRGPU_CUDA(cudaStreamWaitEvent(o.osc_stream, o.ev_mix, 0));
    const int count = (int)(o.osc_produced - o.osc_consumed);
    SDRGPU_TRY(launch_changes(list, [&](const OffsetChanges &c) {
        osc_reproduce_kernel<<<(c.n + 31) / 32, 32, 0, o.osc_stream>>>(o.d_mix, o.d_mix_state, o.d_osc, o.osc_ring_len,
                                                                       o.osc_consumed, count, o.d_held, c);
    }));
    SDRGPU_CUDA(cudaEventRecord(o.ev_osc, o.osc_stream));
    o.osc_pending = true;
    o.osc_safe = o.osc_consumed;
    return SDRGPU_OK;
}

}  // namespace

sdrgpu_status sdrgpu::outputs_select(ChanOutputs &o, const std::vector<sdrgpu_output_channel> &channels, int M,
                                     double sample_rate, int max_blocks, OutputRows *rows)
{
    std::vector<PostChannel> post;
    std::vector<MixChannel> mix;
    std::vector<int> post_of, mix_of;
    int n_two = 0;
    plan_outputs(channels, M, sample_rate, rows, &post, &mix, &post_of, &mix_of, &n_two);

    SDRGPU_CUDA(free_buffers(o));
    o.max_blocks = max_blocks;
    o.n_post = 0;
    o.n_mix = 0;
    // every channel holds the Oscillator's starting phasor until it first mixes (Oscillator.java:24)
    SDRGPU_TRY(upload(&o.d_held, std::vector<float2>(channels.size(), make_float2(0.0f, -1.0f))));
    if (!post.empty()) {
        SDRGPU_TRY(upload(&o.d_post, post));
        SDRGPU_TRY(upload(&o.d_post_state, std::vector<PostState>(post.size(), post_init())));
        SDRGPU_CUDA(cudaMalloc(&o.d_out2, sizeof(float) * 2 * (size_t)max_blocks * (size_t)n_two));
    }
    if (!mix.empty()) {
        SDRGPU_TRY(ensure_osc_stream(o));
        // two calls' worth: a pipeline tops the ring up at the START of a call, for the call after it (outputs_ahead)
        o.osc_ring_len = (2 * max_blocks + 8 + 1) & ~1;   // even: the producer stores pairs
        SDRGPU_TRY(upload(&o.d_mix, mix));
        SDRGPU_TRY(upload(&o.d_mix_state, std::vector<float2>(mix.size(), make_float2(0.0f, -1.0f))));   // Oscillator.java:24
        SDRGPU_CUDA(cudaMalloc(&o.d_osc, sizeof(float2) * mix.size() * (size_t)o.osc_ring_len));
    }
    o.n_post = (int)post.size();
    o.n_mix = (int)mix.size();
    o.post_of = post_of;
    o.mix_of = mix_of;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu::outputs_update(ChanOutputs &o, const std::vector<sdrgpu_output_channel> &old,
                                     const std::vector<sdrgpu_output_channel> &channels, const std::vector<int> &previous,
                                     int M, double sample_rate, cudaStream_t stream, OutputRows *rows)
{
    std::vector<PostChannel> post;
    std::vector<MixChannel> mix;
    std::vector<int> post_of, mix_of;
    int n_two = 0;
    plan_outputs(channels, M, sample_rate, rows, &post, &mix, &post_of, &mix_of, &n_two);
    const int n = (int)channels.size(), n_old_mix = o.n_mix, n_post = (int)post.size(), n_mix = (int)mix.size();
    // held_from / post_from: each new row's old row (-1: new); mix_to: each old mix row's new mix row and selection index
    std::vector<int> held_from(previous), post_from(n_post, -1);
    std::vector<int2> mix_to(n_old_mix, make_int2(-1, -1));
    std::vector<OffsetChange> restart;   // mix rows whose look-ahead is rewritten from their phasor (osc_reproduce_kernel)
    for (int i = 0; i < n; i++) {
        const int p = previous[i];
        const bool was_mixing = p >= 0 && o.mix_of[p] >= 0;
        if (post_of[i] >= 0 && p >= 0) post_from[post_of[i]] = o.post_of[p];
        if (was_mixing) mix_to[o.mix_of[p]] = make_int2(mix_of[i], i);
        // a channel that starts mixing (a new one included) resumes from its held phasor; one that keeps mixing at a new
        // offset mixes its next block with the phasor the old angle produced
        if (mix_of[i] >= 0 && (!was_mixing || old[p].frequency_offset_hz != channels[i].frequency_offset_hz)) {
            OffsetChange c{};
            c.index = mix_of[i];
            c.held_row = was_mixing ? -1 : i;
            c.angle_i = mix[mix_of[i]].angle_i;
            c.angle_q = mix[mix_of[i]].angle_q;
            restart.push_back(c);
        }
    }

    // the calls in flight read the old tables
    SDRGPU_CUDA(cudaStreamSynchronize(stream));
    if (o.osc_stream) SDRGPU_CUDA(cudaStreamSynchronize(o.osc_stream));
    if (n_old_mix == 0) o.osc_produced = o.osc_consumed;   // no ring: nothing ahead
    if (n_mix > 0) {
        SDRGPU_TRY(ensure_osc_stream(o));
        o.osc_ring_len = (2 * o.max_blocks + 8 + 1) & ~1;   // as outputs_select
    }
    // the new tables in `next`; o keeps the old ones until the carry is done
    ChanOutputs next = o;
    next.d_post = nullptr;
    next.d_post_state = nullptr;
    next.d_out2 = nullptr;
    next.d_mix = nullptr;
    next.d_mix_state = nullptr;
    next.d_osc = nullptr;
    next.d_held = nullptr;
    int *d_held_from = nullptr, *d_post_from = nullptr;
    int2 *d_mix_to = nullptr;
    const auto launch_carry = [&]() -> sdrgpu_status {
        SDRGPU_CUDA(cudaMalloc(&next.d_held, sizeof(float2) * (size_t)n));
        SDRGPU_TRY(upload(&d_held_from, held_from));
        gather_kernel<float2><<<(n + 127) / 128, 128, 0, stream>>>(o.d_held, d_held_from, next.d_held, n,
                                                                    make_float2(0.0f, -1.0f));   // Oscillator.java:24
        count_launch();
        if (n_post > 0) {
            SDRGPU_TRY(upload(&next.d_post, post));
            SDRGPU_TRY(upload(&d_post_from, post_from));
            SDRGPU_CUDA(cudaMalloc(&next.d_post_state, sizeof(PostState) * (size_t)n_post));
            SDRGPU_CUDA(cudaMalloc(&next.d_out2, sizeof(float) * 2 * (size_t)o.max_blocks * (size_t)n_two));
            gather_kernel<PostState><<<(n_post + 127) / 128, 128, 0, stream>>>(o.d_post_state, d_post_from,
                                                                                next.d_post_state, n_post, post_init());
            count_launch();
        }
        if (n_mix > 0) {
            SDRGPU_TRY(upload(&next.d_mix, mix));
            SDRGPU_CUDA(cudaMalloc(&next.d_mix_state, sizeof(float2) * (size_t)n_mix));
            SDRGPU_CUDA(cudaMalloc(&next.d_osc, sizeof(float2) * (size_t)n_mix * (size_t)o.osc_ring_len));
        }
        if (n_old_mix > 0) {
            SDRGPU_TRY(upload(&d_mix_to, mix_to));
            osc_carry_kernel<<<n_old_mix, 128, 0, stream>>>(o.d_mix_state, o.d_osc, d_mix_to, next.d_mix_state, next.d_osc,
                                                            next.d_held, o.osc_ring_len, o.osc_consumed,
                                                            (int)(o.osc_produced - o.osc_consumed));
            count_launch();
        }
        SDRGPU_CUDA(cudaGetLastError());
        return SDRGPU_OK;
    };
    sdrgpu_status st = launch_carry();
    if (st == SDRGPU_OK) {
        const cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) st = fail(SDRGPU_ERR_CUDA, "selection update failed: %s", cudaGetErrorString(e));
    }
    cudaFree(d_held_from);
    cudaFree(d_post_from);
    cudaFree(d_mix_to);
    release_tables(st == SDRGPU_OK ? o : next);
    if (st != SDRGPU_OK) return st;
    next.n_post = n_post;
    next.n_mix = n_mix;
    next.post_of = post_of;
    next.mix_of = mix_of;
    next.osc_pending = false;
    next.osc_safe = next.osc_produced;
    o = next;
    return reproduce(o, restart);
}

sdrgpu_status sdrgpu::outputs_set_offsets(ChanOutputs &o, const std::vector<sdrgpu_output_channel> &old,
                                          const std::vector<sdrgpu_output_channel> &channels,
                                          const std::vector<int> &changed, int M, double sample_rate, cudaStream_t stream,
                                          OutputRows *rows, bool *rows_changed)
{
    *rows_changed = false;
    bool transition = false;
    for (int i : changed)
        if (channels[i].bin2 < 0 && (o.mix_of[i] >= 0) != (channels[i].frequency_offset_hz != 0)) transition = true;
    if (transition) {
        // Rare (typically once per channel, at its first correction): the rows of the filter bank change.  This is a
        // selection update that keeps every channel at its own index.
        std::vector<int> same(channels.size());
        for (size_t i = 0; i < same.size(); i++) same[i] = (int)i;
        *rows_changed = true;
        return outputs_update(o, old, channels, same, M, sample_rate, stream, rows);
    }
    std::vector<OffsetChange> post_list, mix_list;
    for (int i : changed) {
        OffsetChange c{};
        c.held_row = -1;
        osc_angle(channels[i].frequency_offset_hz, M, sample_rate, &c.angle_i, &c.angle_q);
        if (o.post_of[i] >= 0) {
            c.index = o.post_of[i];
            post_list.push_back(c);
        } else if (o.mix_of[i] >= 0) {
            c.index = o.mix_of[i];
            mix_list.push_back(c);
        }
    }
    // two-bin channels: behind the calls already enqueued on the channelizer's stream, which read the old angles
    SDRGPU_TRY(launch_changes(post_list, [&](const OffsetChanges &c) {
        post_angle_kernel<<<(c.n + 127) / 128, 128, 0, stream>>>(o.d_post, c);
    }));
    return reproduce(o, mix_list);
}

sdrgpu_status sdrgpu::outputs_before(ChanOutputs &o, int n_blocks, cudaStream_t stream, const float2 **osc, int *osc_start)
{
    SDRGPU_TRY(ensure_osc(o, n_blocks, stream));
    *osc = o.d_osc;
    *osc_start = (int)(o.osc_consumed % o.osc_ring_len);
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu::outputs_after(ChanOutputs &o, float *out, long long stride, int n_blocks, bool mix_fused,
                                    cudaStream_t stream, float *const *rows, long long col)
{
    if (o.n_post > 0) {
        (rows ? post_channel_kernel<true> : post_channel_kernel<false>)<<<o.n_post, 32, 0, stream>>>(
            out, stride, o.d_out2, 2LL * o.max_blocks, n_blocks, o.d_post, o.d_post_state, o.synth, rows, col);
        count_launch();
        SDRGPU_CUDA(cudaGetLastError());
    }
    if (o.n_mix > 0) {
        if (!mix_fused) {
            SDRGPU_TRY(ensure_osc(o, n_blocks, stream));
            (rows ? osc_mix_kernel<true> : osc_mix_kernel<false>)<<<dim3((n_blocks + 255) / 256, o.n_mix), 256, 0, stream>>>(
                out, stride, o.d_mix, o.d_osc, o.osc_ring_len, o.osc_consumed, n_blocks, rows, col);
            count_launch();
        }
        o.osc_consumed += n_blocks;
        SDRGPU_CUDA(cudaEventRecord(o.ev_mix, stream));
        o.mix_recorded = true;
        // top the ring up to a call's worth on the side stream, behind the kernel that has just read it
        const int top_up = o.max_blocks - (int)(o.osc_produced - o.osc_consumed);
        if (top_up > 0) SDRGPU_TRY(produce_ahead(o, top_up));
        SDRGPU_CUDA(cudaGetLastError());
    }
    return SDRGPU_OK;
}

// At the START of a pipeline's call (before its channelizer kernels) the rings are topped up to two calls' worth, i.e. the
// values of the NEXT call are produced beside this call's channelizer / first FIR launches -- throughput-bound kernels that
// lose little to 200 latency-bound warps -- instead of behind them, beside the demodulator, whose launch time is set by its
// most loaded scheduler (8 tuners, all 6400 channels corrected: see DESIGN.md).
sdrgpu_status sdrgpu::outputs_ahead(ChanOutputs &o, cudaStream_t stream)
{
    if (o.n_mix <= 0 || !o.d_osc) return SDRGPU_OK;
    const int top_up = 2 * o.max_blocks - (int)(o.osc_produced - o.osc_consumed);
    if (top_up <= 0) return SDRGPU_OK;
    // the producer in flight (this call's values) first: ev_osc is about to be re-recorded
    if (o.osc_pending) {
        SDRGPU_CUDA(cudaStreamWaitEvent(stream, o.ev_osc, 0));
        o.osc_pending = false;
        o.osc_safe = o.osc_produced;
    }
    return produce_ahead(o, top_up);
}

void sdrgpu::outputs_destroy(ChanOutputs &o)
{
    free_buffers(o);
    if (o.osc_stream) {
        cudaStreamDestroy(o.osc_stream);
        cudaEventDestroy(o.ev_mix);
        cudaEventDestroy(o.ev_osc);
    }
}
