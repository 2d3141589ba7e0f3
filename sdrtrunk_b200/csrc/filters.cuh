// The channel filters of a bank (filters.cu): the half-band decimation stages and the complex FIR + block AGC, as the
// bank's host code and the fused NBFM kernel (fm.cu) see them.
#pragma once
#include "common.cuh"

namespace sdrgpu {

constexpr int kMaxFirTaps = 512;

struct FirTaps {
    float h[kMaxFirTaps];
};

// The FIR kernels read their taps in whole groups of 8, padded with zeros: the taps a filter of n taps runs, and the
// history its input stream keeps.
__host__ __device__ inline int fir_padded_taps(int n) { return (n + 7) & ~7; }

// the taps of one half-band decimate-by-2 stage (length 4 P - 1 or 11; the odd taps but the centre one are zero)
struct HalfBandTaps {
    float c[64];
    int length;
};

// One stage of the decimation cascade on n_channels rows: out[m] for m < n_out at column out_off of the out rows, from
// 2 n_out new input samples that start at `in`, behind the stage's L - 1 samples of history.
sdrgpu_status halfband_launch(const float2 *in, long long in_stride, float2 *out, long long out_stride, int out_off,
                              int n_out, int n_channels, const HalfBandTaps &taps, cudaStream_t stream);

// what one FIR (+ block AGC) launch filters: n samples of n_channels rows, from column in_off of the input rows (behind
// fir_padded_taps(n_taps) samples of history) to column 0 of the output rows
struct FirLaunch {
    const float2 *in;
    long long in_stride;
    int in_off;
    float2 *out;
    long long out_stride;
    int n;
    int agc_block;    // samples per AGC buffer (<= 1024), the gain is per buffer; 0 = no AGC
    int n_channels;
    const FirTaps *taps;
    int n_taps;
    float gain;
    bool throttle;    // the filters share the GPU with the demodulator of the previous chunk (SDRGPU_TUNE_FIR_CTAS_PER_SM)
    cudaStream_t stream;
};
sdrgpu_status fir_agc_launch(const FirLaunch &a);

}  // namespace sdrgpu
