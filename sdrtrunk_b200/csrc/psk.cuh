// The DQPSK symbol demodulator (psk.cu) as the bank's host code sees it: per-channel states, the loop constants, the
// kernel layout and the launch.
#pragma once
#include "common.cuh"

namespace sdrgpu {

constexpr int kMaxTwice = 64;   // 2 * floor(2 * samples/symbol) <= 128 delay-line entries
constexpr int kPskSlack = 32;   // the FIR/AGC output rows are readable this many samples past the valid data

// the DQPSK loop state (PLL, timing, delay lines) of one channel
struct PskState {
    double phase, freq;
    float sampling_point, detected_sps;
    float2 prev_a, prev_b;   // DD: previous preceding / current sample; Gardner: previous middle / current sample
    float2 gardner_prev_symbol;
    int pointer;
    int pad;
    float delay_i[2 * kMaxTwice];
    float delay_q[2 * kMaxTwice];
};

struct PskConfig {
    double max_freq, alpha, beta;
    float sps_gain, counter_gain, max_sps, min_sps;
    float2 rot[4];  // rotate from +45, +135, -45, -135
    int twice;      // floor(2 * sps)
    int gardner;
    double sc[16];  // sincos_f constants (filled by psk_config_constants)
    double two_pi, wrap_base, neg_limit;
    double sync_correction[3];  // PLLPhaseInversionDetector.mPllCorrection of the 90 CW / 90 CCW / 180 detectors
};

struct SyncState {
    unsigned long long bits;   // the undelayed dibit stream, newest dibit in bits 0-1 (MultiSyncPatternMatcher.mBits
    unsigned bits_high;        //   = the low 48 / 40 bits); psk_kernel keeps 96 bits, psk_wide_kernel 64
    int bit_count;             // mBitCount (starts at 2 * delay: the delay buffer's preloaded D00 dibits); psk_kernel:
                               //   as of the last multiple of 16 symbols, psk_wide_kernel: current
    unsigned index;            // symbols demodulated so far
    unsigned pad;
    unsigned align16[2];       // the ring starts on a 16-byte boundary (copied with 16-byte loads)
    // detectors: ring[i & 255] = event the detector raises at symbol i.  Phase 2 framer (kP2Ring entries): the dibit
    // history, ring[i & 511] = dibit of symbol i; bits_high = mDibitsProcessed, pad = mSynchronized
    unsigned char ring[512];
};

// Which demodulator kernel runs a bank: one warp or half a warp per channel (psk_kernel, lanes 32 / 16), several
// samples per lane (psk_multi_kernel, lanes x per = 16 x 1, 8 x 2, 4 x 3, 2 x 6; early = the decision-directed
// early-window variants) or one thread per channel (psk_wide_kernel, lanes 1).
struct PskLayout {
    enum Family { kWarp, kMulti, kWide };
    Family family;
    int lanes, per;
    bool early;
};

// what one demodulator launch reads and advances: C rows of the FIR/AGC output, C channel states, the dibit rows and
// counts (symbols may be null), the sync detector / framer states, and the per-symbol tap values (tap may be null)
struct PskLaunch {
    const float2 *in;
    long long in_stride;
    int n_samples;
    PskState *states;
    const PskConfig *cfg;   // device copy
    uint8_t *symbols;
    int symbol_stride;
    int *counts;
    int accumulate;   // this launch continues the symbol rows of an earlier chunk of the same call
    int n_channels;
    SyncState *sync;
    double *tap;
    int tap_cap;
    cudaStream_t stream;
};

// Validates the demodulator settings of `cfg` at sample rate fs, builds the loop constants into `p`, and allocates
// and uploads the device config and n_channels fresh channel states (and the interpolator table).
sdrgpu_status psk_create(const sdrgpu_bank_config &cfg, double fs, int n_channels, PskConfig &p, PskConfig **d_cfg,
                         PskState **d_states);
// Resets n_channels sync detector / Phase 2 framer states of kind `sync_kind` to a fresh detector.
sdrgpu_status psk_sync_reset(SyncState *d_sync, int n_channels, int sync_kind);
// The kernel layout of a bank of n_channels channels; forced_lanes = 0 picks it from the bank size, else 32, 16, 8,
// 4, 2 or 1 lanes per channel (mapped to the nearest layout that carries the bank's sync detector).
PskLayout psk_layout(const PskConfig &p, int sync_kind, int n_channels, int forced_lanes);
// The layout of the symbol tap's single-channel re-run: its sync detector state must be in the bank's format.
PskLayout psk_tap_layout(const PskLayout &bank, int sync_kind);
void psk_launch(const PskLayout &layout, const PskConfig &p, int sync_kind, const PskLaunch &a);
// CostasLoop.correctInversion (reset = 0) or reset (reset = 1) of one channel, between buffers
void psk_pll_request(PskState *states, int channel, double correction, double max_freq, int reset, cudaStream_t stream);

}  // namespace sdrgpu
