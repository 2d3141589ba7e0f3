// The per-channel bank (bank.cu) as the fused channelizer -> bank pipeline (pipeline.cu) sees it: the handle, its stream
// buffers and the steps of a process call (plan the outputs, run the chain over assembler buffers, carry what is left,
// finish the outputs).
#pragma once
#include "common.cuh"
#include "filters.cuh"
#include "fm.cuh"
#include "psk.cuh"

namespace sdrgpu {

constexpr int kMaxStages = 10;

struct StreamBuf {
    float2 *d = nullptr;
    int hist = 0;          // samples of history kept in front
    long long stride = 0;  // float2 per channel row
};

}  // namespace sdrgpu

struct sdrgpu_bank {
    int device = 0;
    sdrgpu_bank_config cfg{};
    sdrgpu::FirTaps fir_taps{};
    int n_fir = 0;
    int n_stages = 0;
    sdrgpu::HalfBandTaps stage_taps[sdrgpu::kMaxStages];
    // streams[0] = pending input; streams[i] = output of decimation stage i (input of stage i+1 or the FIR)
    sdrgpu::StreamBuf streams[sdrgpu::kMaxStages + 1];
    float2 *d_y = nullptr;  // FIR / AGC output [C][y_stride]
    long long y_stride = 0;
    int fill = 0;           // pending complex samples per channel in streams[0]
    int max_in = 0, max_blocks = 0;
    sdrgpu::PskState *d_psk = nullptr;
    sdrgpu::PskConfig *d_pskcfg = nullptr;  // device copy of `psk`
    sdrgpu::SyncState *d_sync = nullptr;    // [n_channels] sync detector state (sdrgpu_bank_set_sync_detector)
    int sync_kind = SDRGPU_SYNC_NONE;
    int psk_lanes = 0;              // lanes per channel of the demodulator kernel: 0 = by bank size, else 32 / 16 / 1
    sdrgpu::PskConfig psk{};
    sdrgpu::SquelchState *d_sq = nullptr;
    uint8_t *d_gate = nullptr;
    double *d_sq_threshold = nullptr;   // [n_channels] squelch thresholds, linear power (sdrgpu_bank_set_squelch_threshold)
    bool sq_report = false;             // FM_SQUELCH: a status byte per assembler buffer into `symbols`
    // staging for host I/O
    float2 *d_in = nullptr;
    uint8_t *d_sym = nullptr;
    int sym_cap = 0;
    float *d_demod = nullptr;
    long long demod_cap = 0;
    int *d_counts = nullptr;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // The DQPSK demodulator (one warp per channel, latency bound, ~5 % of the SMs) runs on its own stream so that it
    // overlaps the channelizer / FIR kernels of the next chunk; ev_fir orders it after the FIR output it reads, ev_psk
    // orders everything that reuses its buffers (and the caller-visible outputs) after it.
    cudaStream_t psk_stream = nullptr;
    cudaEvent_t ev_fir = nullptr, ev_psk = nullptr;
    // symbol tap (sdrgpu_bank_set_symbol_tap): one channel's demodulator re-run from a shadow copy of its states
    int tap_channel = -1, tap_cap = 0;
    bool tap_ran = false;   // the current / last process call launched the tap run (else it has no symbols)
    double *d_tap = nullptr;
    sdrgpu::PskState *d_tap_state = nullptr;
    sdrgpu::SyncState *d_tap_sync = nullptr;
    int *d_tap_count = nullptr;
    cudaStream_t tap_stream = nullptr;
    cudaEvent_t ev_tap = nullptr, ev_tap_done = nullptr;
    bool psk_pending = false;
    sdrgpu::KernelTimer t_filter, t_demod;
    // FM banks that nbfm_fused_kernel fits (nbfm_fused_fits): no per-stage streams, the raw history lives in fhist, and
    // whole-buffer device calls are read in place (no append copy)
    bool fused_fm = false;
    sdrgpu::NbfmHistory fhist;
    const float2 *direct_in = nullptr;   // this call's new samples, when they are processed where the caller put them
    long long direct_stride = 0;
};

namespace sdrgpu {

inline bool is_dqpsk(int demod) { return demod == SDRGPU_DEMOD_DQPSK_DECISION || demod == SDRGPU_DEMOD_DQPSK_GARDNER; }
inline int final_rate_divisor(const sdrgpu_bank *b) { return b->cfg.decimation > 0 ? b->cfg.decimation : 1; }
// how many output items per channel one assembler buffer produces
inline int max_out_per_block(const sdrgpu_bank *b) { return b->cfg.block_size / final_rate_divisor(b); }
// floats per channel n_blocks assembler buffers write to `demod`
inline int demod_items_for(const sdrgpu_bank *b, int n_blocks) { return (is_fm(b->cfg.demod) ? 1 : 2) * n_blocks * max_out_per_block(b); }

// Where one process call's outputs go on the device (the caller's device buffers, or staging for host buffers)
struct OutPlan {
    int n_blocks = 0;        // assembler buffers per channel this call will complete
    int demod_items = 0;     // floats per channel written to `demod` by this call
    uint8_t *d_sym = nullptr;   // DQPSK dibits, or FM_SQUELCH statuses (reporting on); else null
    int sym_stride = 0;
    float *d_dem = nullptr;
    long long dem_stride = 0;
    int *d_cnt = nullptr;
};

// The steps of a process call of n_blocks assembler buffers into the outputs `o`: check_outputs before any device work,
// plan_outputs, run_chain + consume (once, or once per chunk), finish_outputs.  finish_outputs' dibit_stream: the stream
// a pipeline already sent the host dibit rows and counts out on (else null).
sdrgpu_status check_outputs(const sdrgpu_bank *b, int n_blocks, const sdrgpu_bank_output &o);
sdrgpu_status plan_outputs(sdrgpu_bank *b, int n_blocks, const sdrgpu_bank_output &o, int out_mem, OutPlan *plan);
sdrgpu_status finish_outputs(sdrgpu_bank *b, const OutPlan &plan, const sdrgpu_bank_output &o, int out_mem,
                             cudaStream_t dibit_stream = nullptr);

// Where a run of the chain sits in its call; a single pass is the one run at the start.
struct ChainRun {
    int done = 0;            // assembler buffers of the call before this run: its outputs continue behind theirs
    long long x_off = 0;     // filters-first: samples into the pending input where the run's buffers start
    bool chunked = false;    // one of several runs: the DQPSK demodulator runs on its own stream and accumulates
};

// Filters and demodulates n_blocks assembler buffers of the pending input into the plan's outputs, leaving the input
// where it is; consume() then drops them: stream 0 keeps its history and the unconsumed remainder, the cascade's streams
// their history.
sdrgpu_status run_chain(sdrgpu_bank *b, const OutPlan &plan, int n_blocks, const ChainRun &run = {});
sdrgpu_status consume(sdrgpu_bank *b, int n_blocks);

}  // namespace sdrgpu
