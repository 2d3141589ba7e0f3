// The channelizer's output stage for "special" channels (outputs.cu): two-bin channels and one-bin channels with a
// frequency offset, the oscillator look-ahead rings of the latter, and the arithmetic pfb2_kernel shares with it when it
// mixes the oscillators in itself.  This is what the channelizer's host code sees.
#pragma once
#include <vector>

#include "common.cuh"

namespace sdrgpu {

constexpr int kMaxSynthEntries = 32;   // serpentine entries (4 floats each): filter.length / 2

struct SynthFilter {
    float f[4 * kMaxSynthEntries];  // taps duplicated for I and Q (TwoChannelSynthesizerM2.init)
    int entries;                     // len / 4
};

// two-bin channel (post_channel_kernel)
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

// one-bin channel with a frequency offset (osc_produce_kernel + osc_mix_kernel, or pfb2_kernel's mixing store)
struct MixChannel {
    int row;
    float angle_i, angle_q;
    double gain;
};

// sdrgpu_chan_set_frequency_offsets: new angles for rows of the d_post / d_mix tables, passed by value to the kernels that
// apply them (so nothing on the host has to outlive a launch queued behind calls in flight)
constexpr int kMaxOffsetChanges = 1024;
struct OffsetChange {
    int index;              // row of d_post / d_mix
    int held_row;           // a one-bin channel that starts mixing: its selection index (its phasor in d_held), else -1
    float angle_i, angle_q;
};
struct OffsetChanges {
    int n;
    OffsetChange c[kMaxOffsetChanges];
};

// AbstractOscillator.mixComplex (J/dsp/mixer/AbstractOscillator.java:102-116): sample v times oscillator value z, every
// product, difference and sum rounded on its own
__device__ __forceinline__ float2 mix_complex(float2 v, float2 z)
{
    const float x = __fsub_rn(__fmul_rn(v.x, z.x), __fmul_rn(v.y, z.y));
    const float y = __fadd_rn(__fmul_rn(v.y, z.x), __fmul_rn(v.x, z.y));
    return make_float2(x, y);
}

// Where channel-layout row c of a call starts.  A channelizer's own rows are contiguous: out + c * stride.  A pipeline
// that routes one channelizer's rows to several banks passes a table instead (ROUTED, the kernels' separate instances):
// rows[c] is that row's place in its bank's pending input, and this call's samples start col floats behind it -- one
// offset for every row, because the banks of a pipeline are kept in step.
template <bool ROUTED>
__device__ __forceinline__ float *channel_row(float *out, long long stride, float *const *rows, long long col, int c)
{
    if constexpr (ROUTED) return rows[c] + col;
    else return out + (size_t)c * stride;
}

struct ChanOutputs {
    int max_blocks = 0;             // blocks one channelizer call can produce: scratch rows and rings are sized for it
    SynthFilter synth{};            // two-bin channels' synthesis filter (sdrgpu_chan_select / _update_selection)
    int n_post = 0;                 // two-bin channels
    PostChannel *d_post = nullptr;
    PostState *d_post_state = nullptr;
    float *d_out2 = nullptr;        // scratch rows of the second bins [n_post][2 * max_blocks]
    // one-bin frequency-corrected channels: oscillator values produced ahead of use on a side stream
    int n_mix = 0, osc_ring_len = 0;
    MixChannel *d_mix = nullptr;
    float2 *d_mix_state = nullptr;  // oscillator vector at the producer's position
    float2 *d_osc = nullptr;        // [n_mix][osc_ring_len]
    long long osc_produced = 0, osc_consumed = 0, osc_safe = 0;   // osc_safe: produced by launches already waited for
    cudaStream_t osc_stream = nullptr;
    cudaEvent_t ev_mix = nullptr, ev_osc = nullptr;
    bool osc_pending = false;
    bool mix_recorded = false;      // ev_mix marks the end of the last kernel that read the rings
    // per selected channel: its row of d_post / d_mix (-1: none), and the phasor a one-bin channel holds while it does not
    // mix (OneChannelOutputProcessor keeps its Oscillator when the offset goes to 0)
    std::vector<int> post_of, mix_of;
    float2 *d_held = nullptr;
};

// What the filter bank writes for a selection: the rows (each channel's first bin, then the second bins of two-bin
// channels as scratch rows) with their gains, and whether every bin 0..M-1 is, in order, a frequency-corrected one-bin
// channel with one float-representable gain (mix_gain): pfb2_kernel can then mix the oscillators in itself.
struct OutputRows {
    std::vector<int> sel;
    std::vector<double> gain;   // 1 for special channels (their stage applies the gain) and scratch rows
    bool mix_identity = false;
    float mix_gain = 0.0f;
};

// Rebuilds the stage for a selection at this sample rate and channel count; restarts every oscillator and synthesizer.
sdrgpu_status outputs_select(ChanOutputs &o, const std::vector<sdrgpu_output_channel> &channels, int M, double sample_rate,
                             int max_blocks, OutputRows *rows);
// A new selection `channels` (the current one is `old`) whose entry i continues the channel at index previous[i] of the
// current selection, or is a new channel (-1).  Waits for the work in flight, then builds the tables for the new
// selection and carries every kept channel's state to its new rows: a two-bin channel's PostState, a one-bin channel's
// held phasor, look-ahead window and producer state.  New channels start as after outputs_select; a kept channel at a
// new offset changes only its angle, as outputs_set_offsets does.  The caller has checked that kept entries keep their
// class (one or two bins) and gain.  Returns the filter bank's rows in *rows.
sdrgpu_status outputs_update(ChanOutputs &o, const std::vector<sdrgpu_output_channel> &old,
                             const std::vector<sdrgpu_output_channel> &channels, const std::vector<int> &previous, int M,
                             double sample_rate, cudaStream_t stream, OutputRows *rows);
// New frequency offsets for the selected channels `changed` (old: the selection with the current offsets, channels: with
// the new ones), from the next call on; calls already enqueued keep the old ones.  Two-bin channels and one-bin channels
// that keep mixing change their angle in stream order and keep their oscillator, synthesizer and look-ahead
// (osc_reproduce_kernel).  A one-bin channel that starts or stops mixing changes the filter bank's rows: that is an
// outputs_update keeping every channel at its index, returning the new rows in *rows (*rows_changed); otherwise *rows is
// untouched.
sdrgpu_status outputs_set_offsets(ChanOutputs &o, const std::vector<sdrgpu_output_channel> &old,
                                  const std::vector<sdrgpu_output_channel> &channels, const std::vector<int> &changed,
                                  int M, double sample_rate, cudaStream_t stream, OutputRows *rows, bool *rows_changed);
// Before a filter bank that mixes the oscillators in: makes the rings hold n_blocks values from osc_consumed on (on
// `stream`) and gives the rings ([n_mix][osc_ring_len]) and the slot of the first value.
sdrgpu_status outputs_before(ChanOutputs &o, int n_blocks, cudaStream_t stream, const float2 **osc, int *osc_start);
// After the filter bank wrote n_blocks blocks to the rows of `out` (or, with a row table, to rows[c] + col: channel_row):
// runs post_channel_kernel and, unless the filter bank mixed them (mix_fused), osc_mix_kernel; then tops the rings up
// behind the mix on the side stream.
sdrgpu_status outputs_after(ChanOutputs &o, float *out, long long stride, int n_blocks, bool mix_fused, cudaStream_t stream,
                            float *const *rows = nullptr, long long col = 0);
// A pipeline's look-ahead (chan_osc_ahead): tops the rings up to two calls' worth now.
sdrgpu_status outputs_ahead(ChanOutputs &o, cudaStream_t stream);
void outputs_destroy(ChanOutputs &o);

}  // namespace sdrgpu
