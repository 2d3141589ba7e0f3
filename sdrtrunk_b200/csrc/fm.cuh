// The FM stage of a bank (fm.cu): power squelch and FM discriminator, either behind the bank's filters or as
// nbfm_fused_kernel, which also runs the decimation cascade and the FIR.  This is what the bank's host code sees.
#pragma once
#include "common.cuh"
#include "filters.cuh"

namespace sdrgpu {

inline bool is_fm(int demod) { return demod == SDRGPU_DEMOD_FM || demod == SDRGPU_DEMOD_FM_SQUELCH; }

// PowerSquelch + FMDemodulator state of one channel
struct SquelchState {
    double output;
    int state;  // 0 ATTACK, 1 DECAY, 2 MUTE, 3 UNMUTE
    int ramp_count;
    float prev_i, prev_q;  // FMDemodulator.mPreviousI/Q
};

// The raw history of a bank that nbfm_fused_kernel runs: a ping-pong of [C][hist0] rows holding the last hist0 input
// samples, the front of the next call's windows.
struct NbfmHistory {
    int hist0 = 0;
    int cur = 0;
    float2 *d[2] = {nullptr, nullptr};
};

// Whether nbfm_fused_kernel runs the FM bank of `cfg` with this decimation cascade and FIR, and the raw history it
// needs (*hist0).
bool nbfm_fused_fits(const sdrgpu_bank_config &cfg, const HalfBandTaps *stages, int n_stages, int n_fir, int *hist0);

// Allocates and uploads n_channels fresh channel states (squelch muted, no previous sample) and their squelch
// thresholds, every one `threshold` (linear power).
sdrgpu_status fm_create(int n_channels, double threshold, SquelchState **d_states, double **d_thresholds);

// Sets the squelch threshold (linear power) of one channel, or of every channel with channel = -1, in stream order:
// the FM launches enqueued after it use the new value.
sdrgpu_status fm_set_threshold(double *d_thresholds, int n_channels, int channel, double threshold, cudaStream_t stream);

// what one FM launch reads and advances
struct FmLaunch {
    const float2 *in;          // fused: the new channel-rate samples; else the FIR output
    long long in_stride;
    int n;                     // samples per channel in `in`
    int n_channels;
    int squelch;               // SquelchingFMDemodulator (else FMDemodulator: every sample demodulated)
    double alpha;
    const double *thresholds;  // [C] squelch thresholds (linear power)
    int ramp;
    float gain;
    SquelchState *states;
    float *out;                // [C][n / decimation] demodulated floats, may be null
    long long out_stride;
    uint8_t *status;           // with squelch, may be null: [C][status_stride] one squelch status byte per assembler
    long long status_stride;   // buffer (SDRGPU_SQUELCH_*: state after its last sample | CHANGED)
    int buffer_out;            // demodulated samples per assembler buffer
    uint8_t *gate;             // without `fused`, with squelch: [C][in_stride] gate bytes
    NbfmHistory *fused;        // non-null: nbfm_fused_kernel filters `in` behind this history and flips it
    int n_stages;              // the fused kernel's decimation cascade and FIR
    const HalfBandTaps *stages;
    const FirTaps *fir;
    int n_fir;
    float fir_gain;
    cudaStream_t stream;
};
sdrgpu_status fm_launch(const FmLaunch &a);

}  // namespace sdrgpu
