// The channelizer's output stage for "special" channels: two-bin channels (post_channel_kernel) and one-bin channels with
// a frequency offset (osc_produce_kernel + osc_mix_kernel, or pfb2_kernel mixing the oscillators in where it stores).
// The filter bank leaves their rows at gain 1 (bin values after the 1/M of the inverse FFT); this stage finishes them in
// place on the channelizer's stream.
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
__global__ void __launch_bounds__(32) osc_produce_kernel(const MixChannel *__restrict__ chans, float2 *__restrict__ state,
                                                           float2 *__restrict__ ring, int ring_len, long long start, int count,
                                                           int n_mix)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_mix) return;
    const float2 angle = make_float2(chans[ch].angle_i, chans[ch].angle_q);
    float2 cur = state[ch];
    float2 *r = ring + (size_t)ch * ring_len;
    int pos = (int)(start % ring_len);
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
    state[ch] = cur;
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

// the stage's buffers, once the producer is done with them; the rings restart empty
cudaError_t free_buffers(ChanOutputs &o)
{
    const cudaError_t e = o.osc_stream ? cudaStreamSynchronize(o.osc_stream) : cudaSuccess;
    release(o.d_post);
    release(o.d_post_state);
    release(o.d_out2);
    release(o.d_mix);
    release(o.d_mix_state);
    release(o.d_osc);
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

}  // namespace

sdrgpu_status sdrgpu::outputs_select(ChanOutputs &o, const std::vector<sdrgpu_output_channel> &channels, int M,
                                     double sample_rate, int max_blocks, OutputRows *rows)
{
    const int n = (int)channels.size();
    std::vector<int> &sel = rows->sel;
    std::vector<double> &gd = rows->gain;
    sel.clear();
    gd.clear();
    std::vector<PostChannel> post;
    std::vector<MixChannel> mix;
    int n_two = 0;
    for (int i = 0; i < n; i++) {
        const sdrgpu_output_channel &c = channels[i];
        const bool special = c.bin2 >= 0 || c.frequency_offset_hz != 0;
        sel.push_back(c.bin1);
        // special rows leave the filter bank at gain 1; this stage applies the gain after mixing
        gd.push_back(special ? 1.0 : c.gain);
        if (special) {
            PostChannel pc{};
            pc.row = i;
            pc.row2 = c.bin2 >= 0 ? n_two++ : -1;
            // TwoChannelOutputProcessor mixes unconditionally, OneChannelOutputProcessor only with an offset
            pc.mix = 1;
            // Oscillator.update: anglePerSample = (float)(2 pi f / fs); Complex.fromAngle(float) -> (float)cos, (float)sin
            const double channel_rate = 2.0 * sample_rate / (double)M;
            const float angle = (float)(2.0 * 3.14159265358979323846 * (double)c.frequency_offset_hz / channel_rate);
            pc.angle_i = (float)cos((double)angle);
            pc.angle_q = (float)sin((double)angle);
            pc.gain = c.gain;
            if (c.bin2 >= 0) post.push_back(pc);                                        // two-bin: post_channel_kernel
            else mix.push_back(MixChannel{pc.row, pc.angle_i, pc.angle_q, pc.gain});    // one bin + offset: look-ahead
        }
    }
    for (int i = 0; i < n; i++)
        if (channels[i].bin2 >= 0) {   // scratch rows: the second bins, gain 1
            sel.push_back(channels[i].bin2);
            gd.push_back(1.0);
        }
    rows->mix_identity = (int)mix.size() == n && n == M && (int)sel.size() == n;
    for (size_t m = 0; m < mix.size() && rows->mix_identity; m++)
        if (mix[m].row != (int)m || sel[m] != (int)m || mix[m].gain != mix[0].gain || (double)(float)mix[m].gain != mix[m].gain)
            rows->mix_identity = false;
    rows->mix_gain = mix.empty() ? 0.0f : (float)mix[0].gain;

    SDRGPU_CUDA(free_buffers(o));
    o.max_blocks = max_blocks;
    o.n_post = 0;
    o.n_mix = 0;
    if (!post.empty()) {
        std::vector<PostState> init(post.size());
        std::memset(init.data(), 0, sizeof(PostState) * init.size());
        for (auto &st : init) {
            st.cur_i = 0.0f;   // Oscillator.java:24: mCurrentAngle = new Complex(0.0f, -1.0f)
            st.cur_q = -1.0f;
            st.top_block = 1;  // TwoChannelSynthesizerM2: mTopBlockIndicator = true
        }
        SDRGPU_TRY(upload(&o.d_post, post));
        SDRGPU_TRY(upload(&o.d_post_state, init));
        SDRGPU_CUDA(cudaMalloc(&o.d_out2, sizeof(float) * 2 * (size_t)max_blocks * (size_t)n_two));
    }
    if (!mix.empty()) {
        if (!o.osc_stream) {
            SDRGPU_CUDA(cudaStreamCreateWithFlags(&o.osc_stream, cudaStreamNonBlocking));
            SDRGPU_CUDA(cudaEventCreateWithFlags(&o.ev_mix, cudaEventDisableTiming));
            SDRGPU_CUDA(cudaEventCreateWithFlags(&o.ev_osc, cudaEventDisableTiming));
        }
        // two calls' worth: a pipeline tops the ring up at the START of a call, for the call after it (outputs_ahead)
        o.osc_ring_len = (2 * max_blocks + 8 + 1) & ~1;   // even: the producer stores pairs
        SDRGPU_TRY(upload(&o.d_mix, mix));
        SDRGPU_TRY(upload(&o.d_mix_state, std::vector<float2>(mix.size(), make_float2(0.0f, -1.0f))));   // Oscillator.java:24
        SDRGPU_CUDA(cudaMalloc(&o.d_osc, sizeof(float2) * mix.size() * (size_t)o.osc_ring_len));
    }
    o.n_post = (int)post.size();
    o.n_mix = (int)mix.size();
    return SDRGPU_OK;
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
