// The fused channelizer -> bank pipeline (sdrgpu_pipeline_*): one or several tuners' channelizers write their selected
// channels straight behind the pending samples of one bank, or, routed, of several banks, and the banks' chains
// (bank.cuh) run behind them.  A call runs one of three schedules:
//   run_single_pass     the channelizers over the whole call, then every bank's chain once
//   run_filters_first   device-resident input: the channelizers over the whole call, then FIR / AGC and the DQPSK
//                       demodulator chunk by chunk; asynchronous calls (submit / wait) are left in flight here
//   run_chunked         host input: the whole chain chunk by chunk, the H2D copies hidden behind the kernels
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <vector>

#include "bank.cuh"

using namespace sdrgpu;

struct sdrgpu_pipeline {
    // one or several tuners' channelizers feed consecutive row ranges of ONE bank: the serial demodulator then runs
    // over all their channels in a single launch (it needs thousands of channels to fill the GPU, a tuner has hundreds).
    // A routed pipeline feeds several banks (decoder types) from the same channelizer pass: each selected channel goes
    // to the bank its route names.
    std::vector<sdrgpu_channelizer *> chans;
    std::vector<int> sel;    // channels each channelizer selected when the route was built
    std::vector<sdrgpu_bank *> banks;   // banks[0]'s stream is the pipeline's; the others run on it while the pipeline lives
    std::vector<void *> bank_streams;   // the streams banks[1..] had before (nullptr: their own), restored at destroy
    std::vector<int> row0;   // one bank: first bank row of each channelizer
    std::vector<float **> d_rows;   // several banks: each channelizer's row table (channel_row): row c's place in its bank's pending input
    int chunks = 8;          // host input: a call is cut into time chunks of 1/chunks of its length, after a ramp of smaller ones (1 = single pass)
    int device_chunks = 0;   // device-resident input: no copy to hide, but the demodulator of chunk i still overlaps the filters of chunk i+1 (0 = by bank size)
    // asynchronous calls (sdrgpu_pipeline_submit_multi / _wait): at most two in flight, ev_done[slot] fires when a call's
    // outputs are on the host and its input buffers are no longer read
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_counts[2] = {nullptr, nullptr}, ev_tail = nullptr, ev_h2d = nullptr;
    int inflight = 0, next_slot = 0;
    // copy streams (ensure_copy_streams): host input goes to the device on copy_in, host dibit rows of bank j leave on
    // copy_out[j]
    cudaStream_t copy_in = nullptr;
    cudaEvent_t copy_events[8] = {};
    std::vector<cudaStream_t> copy_out;
};

namespace {

// SDRGPU_TRACE=1: timeline of one chunked pipeline call (events on the copy / filter / demodulator streams, printed to stderr
// relative to the call's first event) -- the tool behind the chunk-size and overlap choices, off by default
struct CallTrace {
    struct Mark { const char *what; int chunk; cudaEvent_t ev; };
    std::vector<Mark> marks;
    bool on = [] { static const bool env = getenv("SDRGPU_TRACE") && atoi(getenv("SDRGPU_TRACE")) != 0; return env; }();
    void mark(const char *what, int chunk, cudaStream_t s)
    {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        marks.push_back({what, chunk, e});
    }
    void dump()
    {
        if (!on || marks.empty()) return;
        cudaDeviceSynchronize();
        for (auto &m : marks) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, marks[0].ev, m.ev);
            fprintf(stderr, "[sdrgpu trace] %-10s chunk %2d  %8.3f ms\n", m.what, m.chunk, ms);
        }
        for (auto &m : marks) cudaEventDestroy(m.ev);
        marks.clear();
    }
};

// The lengths of a call's time chunks, in samples: the first chunk is `first` units of `unit` samples, and the chunks
// double until they are `full` units long (and stop doubling there: a long call has more chunks than an int has bits).
// With `taper`, the last full chunk's worth of the call is cut into halves, in whole units, down to an eighth of a full
// chunk.
struct ChunkRamp {
    int size, full, unit;
    bool taper;
    int next(int left)   // the next chunk of a call with `left` samples to go
    {
        const int want = (size < full ? size : full) * unit;
        if (size < full) size *= 2;
        int n = left < want ? left : want;
        if (taper && size >= full && left <= full * unit) {
            int floor_units = full / 8;
            if (floor_units < 1) floor_units = 1;
            const int left_units = (left + unit - 1) / unit;
            if (left_units > floor_units) {
                int take = (left_units + 1) / 2;
                if (take < floor_units) take = floor_units;
                if ((long long)take * unit < n) n = take * unit;
            }
        }
        return n;
    }
};

// One bank's part of a pipeline call: its outputs, the schedule it would run alone, and how far it has got
struct BankCall {
    sdrgpu_bank *b = nullptr;
    sdrgpu_bank_output out{};
    OutPlan plan;
    int chunk_blocks = 0;        // 1/parts of the call, in whole assembler buffers
    bool single = true;          // one pass over the call
    bool filters_first = false;  // cut, device input, DQPSK, no decimation cascade: FIR / demodulator chunks behind one channelizer pass
    int done = 0;                // assembler buffers of the call the chain has run over
    int dibit_lo = 0;            // host dibit rows streamed chunk by chunk: columns below are final and on the host
    cudaStream_t copy_out = nullptr;   // the stream host dibit rows stream out on chunk by chunk (null: they leave at the end)
    bool dibits_streamed = false;
};

// One pipeline call, as its schedule sees it
struct Call {
    const void *const *iq;
    int n_floats, in_mem, out_mem;
    int n_samples;               // samples per channel the channelizers complete
    bool async;
    std::vector<BankCall> banks;
    CallTrace trace;
};

// calls in flight complete on the device before a synchronous path touches what they use (their bookkeeping -- the
// caller's sdrgpu_pipeline_wait -- is unchanged)
sdrgpu_status pipeline_drain(sdrgpu_pipeline *p)
{
    for (int i = 0; i < 2; i++)
        if (p->ev_done[i]) SDRGPU_CUDA(cudaEventSynchronize(p->ev_done[i]));
    return SDRGPU_OK;
}

// the copy streams and the events of asynchronous calls, made by the first call that copies to or from the host (ev_h2d
// is made last: a call after a failed attempt makes what is missing)
sdrgpu_status ensure_copy_streams(sdrgpu_pipeline *p)
{
    if (p->ev_h2d) return SDRGPU_OK;
    if (!p->copy_in) SDRGPU_CUDA(cudaStreamCreateWithFlags(&p->copy_in, cudaStreamNonBlocking));
    for (auto &s : p->copy_out)
        if (!s) SDRGPU_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    for (auto &e : p->copy_events)
        if (!e) SDRGPU_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (cudaEvent_t *e : {&p->ev_done[0], &p->ev_done[1], &p->ev_counts[0], &p->ev_counts[1], &p->ev_tail, &p->ev_h2d})
        if (!*e) SDRGPU_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    return SDRGPU_OK;
}

// Every argument and state check of a call, made before anything is staged, swapped or enqueued: a refused call changes
// nothing.  The chunked schedules drive the channelizer internals directly, so these include the checks
// sdrgpu_chan_process makes for a single call.
sdrgpu_status check_call(const sdrgpu_pipeline *p, const void *const *iq, int n_floats, const sdrgpu_bank_output *outputs)
{
    if (n_floats < 0 || n_floats % 2 != 0) return fail(SDRGPU_ERR_INVALID_ARG, "n_floats must be even (interleaved I/Q)");
    const int K = (int)p->chans.size();
    if (n_floats > 0) {
        if (!iq) return fail(SDRGPU_ERR_INVALID_ARG, "iq is NULL");
        for (int k = 0; k < K; k++)
            if (!iq[k]) return fail(SDRGPU_ERR_INVALID_ARG, "iq[%d] is NULL", k);
    }
    for (int k = 0; k < K; k++) {
        if (n_floats / 2 > sdrgpu::chan_max_in(p->chans[k]))
            return fail(SDRGPU_ERR_OVERFLOW, "input of %d floats exceeds channelizer %d's max_input_floats %d", n_floats, k,
                        2 * sdrgpu::chan_max_in(p->chans[k]));
        if (sdrgpu::chan_leftover(p->chans[k]) != sdrgpu::chan_leftover(p->chans[0]))
            return fail(SDRGPU_ERR_BAD_STATE, "channelizer %d is not in step with channelizer 0 (feed all tuners of a pipeline "
                                              "the same number of samples)", k);
        if (sdrgpu::chan_selected_count(p->chans[k]) != p->sel[(size_t)k])
            return fail(SDRGPU_ERR_BAD_STATE, "channelizer %d selects %d channels, the pipeline was built for %d", k,
                        sdrgpu::chan_selected_count(p->chans[k]), p->sel[(size_t)k]);
    }
    // the channelizers write their channel layout straight behind the banks' pending samples
    const int n = sdrgpu_chan_blocks_for(p->chans[0], n_floats);
    for (size_t j = 0; j < p->banks.size(); j++) {
        const sdrgpu_bank *bk = p->banks[j];
        if (n > bk->max_in)
            return fail(SDRGPU_ERR_OVERFLOW, "%d samples per channel exceed the bank's max_samples_per_call %d", n, bk->max_in);
        SDRGPU_TRY(check_outputs(bk, (bk->fill + n) / bk->cfg.block_size, outputs[j]));
    }
    return SDRGPU_OK;
}

// one bank: where tuner k's rows of a call go, behind the pending samples of the bank's rows row0[k]..
float *bank_rows(const sdrgpu_pipeline *p, int k)
{
    const StreamBuf &s0 = p->banks[0]->streams[0];
    return reinterpret_cast<float *>(s0.d + (size_t)p->row0[k] * s0.stride + s0.hist + p->banks[0]->fill);
}

// n complex samples of tuner k, on the device (d_chunk), through its channelizer behind the banks' pending samples
// (routed: through the tuner's row table, at the banks' common column)
sdrgpu_status channelize_chunk(sdrgpu_pipeline *p, int k, const float2 *d_chunk, int n, int *got)
{
    const sdrgpu_bank *b = p->banks[0];
    if (p->banks.size() == 1)
        return sdrgpu::chan_enqueue(p->chans[k], d_chunk, n, bank_rows(p, k), 2 * b->streams[0].stride, SDRGPU_LAYOUT_CHANNELS, got);
    return sdrgpu::chan_enqueue(p->chans[k], d_chunk, n, nullptr, 0, SDRGPU_LAYOUT_CHANNELS, got, p->d_rows[(size_t)k], 2LL * b->fill);
}

// the call's n_floats values of tuner k through its channelizer, written behind the banks' pending samples
sdrgpu_status channelize_call(sdrgpu_pipeline *p, int k, const void *iq, int n_floats, int in_mem, int *got)
{
    sdrgpu_channelizer *chan = p->chans[k];
    if (p->banks.size() == 1)
        return sdrgpu_chan_process(chan, iq, n_floats, in_mem, bank_rows(p, k), 2 * p->banks[0]->streams[0].stride, SDRGPU_DEVICE,
                                   SDRGPU_LAYOUT_CHANNELS, got);
    const int n = n_floats / 2;
    if (n > 0 && in_mem == SDRGPU_HOST) SDRGPU_TRY(sdrgpu::chan_upload(chan, iq, 0, n, sdrgpu::chan_stream(chan)));
    if (n > 0 && in_mem == SDRGPU_DEVICE && ((uintptr_t)iq & 7) != 0 && sdrgpu::chan_complex_bytes(chan) == 8)
        return fail(SDRGPU_ERR_INVALID_ARG, "device input must be 8-byte aligned");
    const float2 *src = sdrgpu::chan_convert(chan, in_mem == SDRGPU_HOST ? nullptr : iq, 0, n);
    if (!src && n > 0) return fail(SDRGPU_ERR_NOMEM, "cannot allocate the channelizer input staging buffer");
    SDRGPU_TRY(channelize_chunk(p, k, src, n, got));
    // the caller's buffer is not read after the call returns (sdrgpu_chan_process synchronises the same way)
    if (n > 0 && in_mem == SDRGPU_HOST) SDRGPU_CUDA(cudaStreamSynchronize(sdrgpu::chan_stream(chan)));
    return SDRGPU_OK;
}

sdrgpu_status plan_call(BankCall &c, const Call &call)
{
    return plan_outputs(c.b, (c.b->fill + call.n_samples) / c.b->cfg.block_size, c.out, call.out_mem, &c.plan);
}

sdrgpu_status finish_call(BankCall &c, const Call &call)
{
    return finish_outputs(c.b, c.plan, c.out, call.out_mem, c.dibits_streamed ? c.copy_out : nullptr);
}

// the chain once over every buffer the call completes (consume is a no-op without any)
sdrgpu_status run_pass(BankCall &c)
{
    if (c.plan.n_blocks > 0) SDRGPU_TRY(run_chain(c.b, c.plan, c.plan.n_blocks));
    return consume(c.b, c.plan.n_blocks);
}

sdrgpu_status run_single_pass(sdrgpu_pipeline *p, Call &call)
{
    if (call.async) SDRGPU_TRY(pipeline_drain(p));
    for (BankCall &c : call.banks) SDRGPU_TRY(plan_call(c, call));
    int got = 0;
    for (int k = 0; k < (int)p->chans.size(); k++)
        SDRGPU_TRY(channelize_call(p, k, call.iq ? call.iq[k] : nullptr, call.n_floats, call.in_mem, &got));
    for (BankCall &c : call.banks) {
        c.b->fill += got;
        SDRGPU_TRY(run_pass(c));
    }
    for (BankCall &c : call.banks) SDRGPU_TRY(finish_call(c, call));
    return SDRGPU_OK;
}

// Device-resident input, filters-first schedule: every tuner's whole buffer goes through its channelizer (one launch per
// tuner), then FIR / AGC and the demodulator run chunk by chunk, the FIR of chunk i+1 beside the demodulator of chunk i.
// The channelizer is kept out of the overlap on purpose: its CTAs need half an SM's registers and shared memory each,
// beside the resident demodulator only one fits per SM and it crawls (measured: 0.35 -> 1.2 ms per quarter call, and the
// step time depended on which kernel reached the SMs first), while the FIR's small CTAs share an SM with the demodulator
// gracefully.  Banks this schedule does not serve run one pass behind the channelizers.
// An asynchronous call shares the dibit / count staging with the call in flight, whose copies to the host run on the
// copy-out stream while this call's channelizers and first FIR launch are already at work: the counts are cleared behind
// that call's (small, first) counts copy, the first demodulator launch waits for its dibit rows.  *went_async: the call
// was left in flight, its completion event recorded in ev_done[next_slot].
sdrgpu_status run_filters_first(sdrgpu_pipeline *p, Call &call, bool *went_async)
{
    sdrgpu_bank *b = p->banks[0];
    const int K = (int)p->chans.size();
    const int block = b->cfg.block_size;
    const bool gate = call.async && p->inflight > 0;
    const int prev_slot = p->next_slot ^ 1;
    BankCall &c0 = call.banks[0];
    if (call.async && (b->fill + call.n_samples) / block > 0 && c0.out.symbol_stride > b->sym_cap)
        SDRGPU_TRY(pipeline_drain(p));   // plan_outputs reallocates
    for (BankCall &c : call.banks) SDRGPU_TRY(plan_call(c, call));
    if (gate) SDRGPU_CUDA(cudaStreamWaitEvent(b->stream, p->ev_counts[prev_slot], 0));
    for (BankCall &c : call.banks)
        if (c.filters_first)
            SDRGPU_CUDA(cudaMemsetAsync(c.plan.d_cnt, 0, sizeof(int) * (size_t)c.b->cfg.n_channels, b->stream));
    // frequency-corrected channels: every tuner's oscillator producer for the NEXT call starts now, beside the
    // channelizers, and is done (or nearly) when the first demodulator launch starts
    CallTrace &trace = call.trace;
    trace.mark("start", 0, b->stream);
    for (int k = 0; k < K; k++) SDRGPU_TRY(sdrgpu::chan_osc_ahead(p->chans[k]));
    for (int k = 0; k < K; k++)
        if (sdrgpu::chan_osc_stream(p->chans[k])) trace.mark("osc", k, sdrgpu::chan_osc_stream(p->chans[k]));
    int got = 0;
    for (int k = 0; k < K; k++) {
        SDRGPU_TRY(channelize_call(p, k, call.iq[k], call.n_floats, call.in_mem, &got));
        trace.mark("pfb", k, b->stream);
    }
    for (BankCall &c : call.banks) c.b->fill += got;
    if (gate) SDRGPU_CUDA(cudaStreamWaitEvent(b->stream, p->ev_done[prev_slot], 0));
    for (BankCall &c : call.banks) {
        sdrgpu_bank *bk = c.b;
        if (!c.filters_first) {
            SDRGPU_TRY(run_pass(c));
            continue;
        }
        // the rows stay where the channelizers wrote them until the last chunk; the FIR launch of the first chunk has no
        // demodulator to run beside: it is kept short (a quarter, then half a chunk)
        const int total_nb = bk->fill / block, chunk_nb = c.chunk_blocks / block;
        ChunkRamp ramp{chunk_nb >= 4 ? chunk_nb / 4 : chunk_nb, chunk_nb, 1, false};
        while (c.done < total_nb) {
            const int nb = ramp.next(total_nb - c.done);
            const int chunk_no = c.done / (chunk_nb > 0 ? chunk_nb : 1);
            SDRGPU_TRY(run_chain(bk, c.plan, nb, {c.done, (long long)c.done * block, true}));
            trace.mark("filters", chunk_no, b->stream);
            trace.mark("demod", chunk_no, bk->psk_stream);
            c.done += nb;
        }
        SDRGPU_TRY(consume(bk, total_nb));
    }
    trace.dump();
    const int total_nb = c0.plan.n_blocks;
    uint8_t *symbols = c0.out.symbols;
    const int symbol_stride = c0.out.symbol_stride;
    if (call.async && call.out_mem == SDRGPU_HOST && symbols && !c0.out.demod && total_nb > 0 && c0.plan.d_sym == b->d_sym) {
        // left in flight: counts, then the dibit rows, leave on the copy-out stream behind the last demodulator launch
        // and the bank stream's tail; nothing is synchronised
        cudaStream_t out = p->copy_out[0];
        SDRGPU_CUDA(cudaEventRecord(p->ev_tail, b->stream));
        SDRGPU_CUDA(cudaStreamWaitEvent(out, p->ev_tail, 0));
        if (b->psk_pending) SDRGPU_CUDA(cudaStreamWaitEvent(out, b->ev_psk, 0));
        if (c0.out.counts)
            SDRGPU_CUDA(cudaMemcpyAsync(c0.out.counts, c0.plan.d_cnt, sizeof(int) * (size_t)b->cfg.n_channels,
                                        cudaMemcpyDeviceToHost, out));
        SDRGPU_CUDA(cudaEventRecord(p->ev_counts[p->next_slot], out));
        SDRGPU_CUDA(cudaMemcpy2DAsync(symbols, (size_t)symbol_stride, c0.plan.d_sym, (size_t)c0.plan.sym_stride,
                                      (size_t)symbol_stride, (size_t)b->cfg.n_channels, cudaMemcpyDeviceToHost, out));
        SDRGPU_CUDA(cudaEventRecord(p->ev_done[p->next_slot], out));
        *went_async = true;
        return SDRGPU_OK;
    }
    for (BankCall &c : call.banks) SDRGPU_TRY(finish_call(c, call));
    return SDRGPU_OK;
}

// The tuner buffers are processed in time chunks: the H2D copy of chunk i+1 (host input) and its channelizer / FIR
// kernels overlap the demodulator of chunk i, which runs on its own stream.  Every stage carries its state from
// chunk to chunk exactly as from call to call, so the outputs do not depend on the cut; DQPSK symbol rows continue
// where the previous chunk stopped.
sdrgpu_status run_chunked(sdrgpu_pipeline *p, Call &call)
{
    sdrgpu_bank *b = p->banks[0];   // the pipeline's stream is this bank's
    const int K = (int)p->chans.size();
    const int block = b->cfg.block_size;
    const int half = sdrgpu::chan_half(p->chans[0]);
    if (call.async) SDRGPU_TRY(pipeline_drain(p));   // (a bank the filters-first schedule does not serve: this call runs to completion)
    if (call.in_mem == SDRGPU_HOST || call.out_mem == SDRGPU_HOST) SDRGPU_TRY(ensure_copy_streams(p));
    bool dq_any = false;
    int chunk_blocks = 0;   // the shortest chunk any bank wants
    for (const BankCall &c : call.banks) {
        dq_any |= is_dqpsk(c.b->cfg.demod);
        if (!c.single && (chunk_blocks == 0 || c.chunk_blocks < chunk_blocks)) chunk_blocks = c.chunk_blocks;
    }
    // Host dibit rows leave chunk by chunk on their own stream instead of as one copy behind the last demodulator launch
    // (40 MB for 6400 channels x 1 s: 0.8 ms of the step).  A row's symbol count after n samples lies between
    // n / (max_sps + 0.3 counter_gain) and n / (min_sps - 0.3 counter_gain) (InterpolatingSampleBuffer clamps the detected
    // samples per symbol, the timing error is clipped to +/- 0.3), so after every chunk the columns [lo, hi) are copied with
    // lo <= every row's count at the previous chunk (everything below is final and already on the host) and hi >= every row's
    // count now; the windows overlap and later copies carry the final values.
    for (size_t j = 0; j < call.banks.size(); j++) {
        BankCall &c = call.banks[j];
        SDRGPU_TRY(plan_call(c, call));
        if (is_dqpsk(c.b->cfg.demod))
            SDRGPU_CUDA(cudaMemsetAsync(c.plan.d_cnt, 0, sizeof(int) * (size_t)c.b->cfg.n_channels, b->stream));
        if (is_dqpsk(c.b->cfg.demod) && call.out_mem == SDRGPU_HOST && c.out.symbols != nullptr && c.plan.d_sym != nullptr)
            c.copy_out = p->copy_out[j];
    }
    const int n_in = call.n_floats / 2;
    int done_in = 0, ci = 0;
    CallTrace &trace = call.trace;
    trace.mark("start", 0, b->stream);
    int chunk_no = 0;
    // The demodulator stream is the critical path (it is serial and by far the longest stage), so it has to start as
    // early as possible: the first chunk is a single assembler buffer and the chunks double until they reach
    // 1/chunks of the call (measured on B200, 400 C4FM channels, 0.98 s of signal: 2.83 -> 2.77 ms per call).
    // ... and it has to end as soon as possible after the last byte has arrived: what is left once the last H2D copy
    // has landed is that chunk's whole chain, so the last full chunk of a call is cut into halves down to an eighth
    // of a chunk.
    const bool host_dq = dq_any && call.in_mem == SDRGPU_HOST;
    ChunkRamp ramp{host_dq ? 1 : chunk_blocks / block, chunk_blocks / block, block * half, host_dq};
    while (done_in < n_in) {
        const int n = ramp.next(n_in - done_in);
        int got = 0;
        for (int k = 0; k < K; k++) {
            sdrgpu_channelizer *chan = p->chans[k];
            const float2 *d_chunk;
            if (call.in_mem == SDRGPU_HOST) {
                cudaEvent_t ev = p->copy_events[ci % 8];
                SDRGPU_TRY(sdrgpu::chan_upload(chan, call.iq[k], (size_t)done_in, n, p->copy_in));
                SDRGPU_CUDA(cudaEventRecord(ev, p->copy_in));
                SDRGPU_CUDA(cudaStreamWaitEvent(b->stream, ev, 0));
                if (k == K - 1) trace.mark("h2d", chunk_no, p->copy_in);
                d_chunk = sdrgpu::chan_convert(chan, nullptr, (size_t)done_in, n);
                ci++;
            } else {
                d_chunk = sdrgpu::chan_convert(chan, call.iq[k], (size_t)done_in, n);
            }
            if (!d_chunk) return fail(SDRGPU_ERR_NOMEM, "cannot allocate the channelizer input staging buffer");
            sdrgpu::chan_set_throttled(chan, dq_any && done_in > 0);   // a demodulator launch of an earlier chunk is running
            const sdrgpu_status st = channelize_chunk(p, k, d_chunk, n, &got);
            sdrgpu::chan_set_throttled(chan, false);
            SDRGPU_TRY(st);
        }
        for (BankCall &c : call.banks) c.b->fill += got;
        trace.mark("pfb", chunk_no, b->stream);
        for (BankCall &c : call.banks) {
            sdrgpu_bank *bk = c.b;
            const int nb = bk->fill / block;
            if (nb <= 0) continue;
            SDRGPU_TRY(run_chain(bk, c.plan, nb, {c.done, 0, true}));
            SDRGPU_TRY(consume(bk, nb));
            c.done += nb;
            trace.mark("filters", chunk_no, b->stream);
            if (is_dqpsk(bk->cfg.demod)) trace.mark("demod", chunk_no, bk->psk_stream);
            const long long y_off = (long long)c.done * max_out_per_block(bk);
            const double spacing_max = (double)bk->psk.max_sps + 0.3 * fabs((double)bk->psk.counter_gain) + 1e-3;
            const double spacing_min = (double)bk->psk.min_sps - 0.3 * fabs((double)bk->psk.counter_gain) - 1e-3;
            if (c.copy_out && spacing_min > 1.0) {
                const int symbol_stride = c.out.symbol_stride;
                int hi = (int)((double)y_off / spacing_min) + 8;
                if (hi > symbol_stride) hi = symbol_stride;
                if (hi > c.dibit_lo) {
                    SDRGPU_CUDA(cudaStreamWaitEvent(c.copy_out, bk->ev_psk, 0));   // recorded behind this chunk's demodulator
                    SDRGPU_CUDA(cudaMemcpy2DAsync(c.out.symbols + c.dibit_lo, (size_t)symbol_stride, c.plan.d_sym + c.dibit_lo,
                                                  (size_t)c.plan.sym_stride, (size_t)(hi - c.dibit_lo), (size_t)bk->cfg.n_channels,
                                                  cudaMemcpyDeviceToHost, c.copy_out));
                }
                int lo = (int)((double)y_off / spacing_max) - 8;
                if (lo > hi) lo = hi;
                if (lo > c.dibit_lo) c.dibit_lo = lo;
                c.dibits_streamed = true;
                trace.mark("d2h", chunk_no, c.copy_out);
            }
        }
        done_in += n;
        chunk_no++;
    }
    for (BankCall &c : call.banks) {
        if (c.dibits_streamed && c.out.counts) {
            SDRGPU_CUDA(cudaStreamWaitEvent(c.copy_out, c.b->ev_psk, 0));
            SDRGPU_CUDA(cudaMemcpyAsync(c.out.counts, c.plan.d_cnt, sizeof(int) * (size_t)c.b->cfg.n_channels, cudaMemcpyDeviceToHost,
                                        c.copy_out));
        }
    }
    for (BankCall &c : call.banks) SDRGPU_TRY(finish_call(c, call));
    // The library never keeps a caller pointer after the call returns (sdrgpu.h): with host input the H2D copies read
    // `iq` until the last chunk's event fires, and the staging they fill is reused by the next call.  b->stream waits on
    // every copy event, so draining it covers the copy stream as well.
    if (call.in_mem == SDRGPU_HOST) SDRGPU_CUDA(cudaStreamSynchronize(b->stream));
    trace.dump();
    return SDRGPU_OK;
}

// A checked call (check_call): picks the schedule.  An asynchronous call (went_async not null: sdrgpu_pipeline_submit_multi,
// which has put the host buffers into the channelizers' staging and passes that as device-resident input): a
// filters-first DQPSK call is left in flight -- *went_async = true -- every other shape of call runs to completion as
// usual.  Only one-bank pipelines are called so.
sdrgpu_status process_call(sdrgpu_pipeline *p, const void *const *iq, int n_floats, int in_mem, const sdrgpu_bank_output *outputs,
                           int out_mem, bool *went_async)
{
    const bool async = went_async != nullptr;
    sdrgpu_bank *b = p->banks[0];
    for (sdrgpu_channelizer *chan : p->chans) SDRGPU_TRY(sdrgpu_chan_set_stream(chan, b->stream));
    const int block = b->cfg.block_size;
    const int n_samples = sdrgpu_chan_blocks_for(p->chans[0], n_floats);
    Call call{iq, n_floats, in_mem, out_mem, n_samples, async, std::vector<BankCall>(p->banks.size()), {}};
    // Each bank runs the schedule it would run alone.  Chunks of whole assembler buffers: 1/chunks of the call, at least
    // one buffer per channel.  Device-resident input has no copy to hide: a bank large enough that its demodulator launch
    // fills the schedulers (several tuners) is run in six time chunks behind a ramp (B200, 8 x 800 channels: 6.19 ms with
    // four equal chunks, 6.0 ms so; one pass 6.6 ms); a single tuner's bank is latency bound either way and saves the
    // extra launches (each extra chunk costs ~30 us of launch / prologue time)
    bool all_single = true, any_filters_first = false;
    for (size_t j = 0; j < call.banks.size(); j++) {
        BankCall &c = call.banks[j];
        c.b = p->banks[j];
        c.out = outputs[j];
        const int auto_parts = c.b->cfg.n_channels >= 2400 ? 6 : 1;
        const int want_parts = in_mem == SDRGPU_HOST ? p->chunks : (p->device_chunks > 0 ? p->device_chunks : auto_parts);
        const int parts = want_parts > 1 ? want_parts : 1;
        c.chunk_blocks = ((n_samples + parts - 1) / parts + block - 1) / block * block;
        const bool ff = in_mem == SDRGPU_DEVICE && is_dqpsk(c.b->cfg.demod) && c.b->n_stages == 0 && !c.b->fused_fm;
        const bool stay_async = async && ff && n_floats > 0 && (c.b->fill + n_samples) / block > 0;   // one chunk is fine there
        c.single = !stay_async && (parts == 1 || n_floats <= 0 || n_samples <= c.chunk_blocks);
        c.filters_first = ff && !c.single;
        all_single &= c.single;
        any_filters_first |= c.filters_first;
    }
    SDRGPU_CUDA(cudaSetDevice(b->device));
    if (all_single) return run_single_pass(p, call);
    if (any_filters_first) return run_filters_first(p, call, went_async);
    return run_chunked(p, call);
}

// the synchronous calls: none may be in flight, and every check comes first
sdrgpu_status process_sync(sdrgpu_pipeline *p, const void *const *iq, int n_floats, int in_mem, const sdrgpu_bank_output *outputs,
                           int out_mem)
{
    if (p->inflight > 0)
        return fail(SDRGPU_ERR_BAD_STATE, "%d asynchronous call(s) in flight: sdrgpu_pipeline_wait first", p->inflight);
    SDRGPU_TRY(check_call(p, iq, n_floats, outputs));
    return process_call(p, iq, n_floats, in_mem, outputs, out_mem, nullptr);
}

}  // namespace

extern "C" {

sdrgpu_status sdrgpu_pipeline_create_routed(sdrgpu_pipeline **out, sdrgpu_channelizer *const *chans, int n_chans,
                                            sdrgpu_bank *const *banks, int n_banks, const int *route)
{
    if (!out || !chans || n_chans <= 0 || !banks || n_banks <= 0 || !route)
        return fail(SDRGPU_ERR_INVALID_ARG, "NULL / empty argument");
    // every check comes before any device work: a refused pipeline leaves the handles as they were
    std::vector<int> sel;
    int rows = 0;
    for (int k = 0; k < n_chans; k++) {
        if (!chans[k]) return fail(SDRGPU_ERR_INVALID_ARG, "channelizer %d is NULL", k);
        // equal channel counts: every tuner then completes the same number of blocks per call, so the bank's rows stay
        // aligned in time (tuners of different rates belong in different banks)
        if (sdrgpu::chan_half(chans[k]) != sdrgpu::chan_half(chans[0]))
            return fail(SDRGPU_ERR_INVALID_ARG, "channelizer %d has a different channel count than channelizer 0", k);
        sel.push_back(sdrgpu::chan_selected_count(chans[k]));
        rows += sel.back();
    }
    for (int j = 0; j < n_banks; j++) {
        if (!banks[j]) return fail(SDRGPU_ERR_INVALID_ARG, "bank %d is NULL", j);
        for (int i = 0; i < j; i++)
            if (banks[i] == banks[j]) return fail(SDRGPU_ERR_INVALID_ARG, "bank %d is listed twice (as bank %d)", j, i);
        // the channelizers complete blocks for all banks at once, and the banks take them in assembler buffers of
        // block_size samples (PolyphaseChannelSource.java:42: 1024 for every preset)
        if (banks[j]->cfg.block_size != banks[0]->cfg.block_size)
            return fail(SDRGPU_ERR_INVALID_ARG, "bank %d has block_size %d, bank 0 %d", j, banks[j]->cfg.block_size,
                        banks[0]->cfg.block_size);
        // the channelizers write one call's samples at one column of every bank: the banks have to be in step
        if (n_banks > 1 && banks[j]->fill != 0)
            return fail(SDRGPU_ERR_BAD_STATE, "bank %d has %d samples pending", j, banks[j]->fill);
    }
    std::vector<int> per_bank((size_t)n_banks, 0);
    for (int r = 0; r < rows; r++) {
        if (route[r] < 0 || route[r] >= n_banks)
            return fail(SDRGPU_ERR_INVALID_ARG, "route[%d] = %d is not a bank index (%d banks)", r, route[r], n_banks);
        per_bank[(size_t)route[r]]++;
    }
    for (int j = 0; j < n_banks; j++)
        if (per_bank[(size_t)j] != banks[j]->cfg.n_channels) {
            if (n_banks == 1)
                return fail(SDRGPU_ERR_INVALID_ARG, "the channelizers select %d channels but the bank has %d", rows,
                            banks[0]->cfg.n_channels);
            return fail(SDRGPU_ERR_INVALID_ARG, "the route gives bank %d %d channels but the bank has %d", j, per_bank[(size_t)j],
                        banks[j]->cfg.n_channels);
        }

    auto *p = new sdrgpu_pipeline();
    p->chans.assign(chans, chans + n_chans);
    p->sel = sel;
    p->banks.assign(banks, banks + n_banks);
    p->copy_out.assign((size_t)n_banks, nullptr);
    int row = 0;
    for (int k = 0; k < n_chans; k++) {
        p->row0.push_back(row);
        row += sel[(size_t)k];
    }
    if (n_banks > 1) {
        // row tables: selected channel c of channelizer k -> the next row of its bank, at that row's history
        std::vector<int> next((size_t)n_banks, 0);
        int r = 0;
        for (int k = 0; k < n_chans; k++) {
            std::vector<float *> table;
            for (int c = 0; c < sel[(size_t)k]; c++, r++) {
                const StreamBuf &s0 = banks[route[r]]->streams[0];
                table.push_back(reinterpret_cast<float *>(s0.d + (size_t)next[(size_t)route[r]]++ * s0.stride + s0.hist));
            }
            float **d = nullptr;
            cudaError_t e = cudaMalloc(&d, sizeof(float *) * table.size());
            if (e == cudaSuccess) e = cudaMemcpy(d, table.data(), sizeof(float *) * table.size(), cudaMemcpyHostToDevice);
            if (d) p->d_rows.push_back(d);
            if (e != cudaSuccess) {
                sdrgpu_pipeline_destroy(p);
                return fail(SDRGPU_ERR_CUDA, "row table upload failed: %s", cudaGetErrorString(e));
            }
        }
        // one stream for the whole pipeline: the channelizers' stores of the next chunk are then ordered behind every
        // bank's carry of this one (the DQPSK demodulators keep their own streams, as in a one-bank pipeline)
        for (int j = 1; j < n_banks; j++) {
            sdrgpu_bank *b = banks[j];
            void *before = b->stream == b->own_stream ? nullptr : (void *)b->stream;
            const sdrgpu_status st = sdrgpu_bank_set_stream(b, banks[0]->stream);
            if (st != SDRGPU_OK) {
                sdrgpu_pipeline_destroy(p);
                return st;
            }
            p->bank_streams.push_back(before);
        }
    }
    *out = p;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_pipeline_create_multi(sdrgpu_pipeline **out, sdrgpu_channelizer *const *chans, int n_chans,
                                           sdrgpu_bank *bank)
{
    if (!out || !chans || n_chans <= 0 || !bank) return fail(SDRGPU_ERR_INVALID_ARG, "NULL / empty argument");
    int rows = 0;
    for (int k = 0; k < n_chans; k++) {
        if (!chans[k]) return fail(SDRGPU_ERR_INVALID_ARG, "channelizer %d is NULL", k);
        rows += sdrgpu::chan_selected_count(chans[k]);
    }
    const std::vector<int> route((size_t)rows + 1, 0);   // (+ 1: never an empty vector's NULL data)
    return sdrgpu_pipeline_create_routed(out, chans, n_chans, &bank, 1, route.data());
}

sdrgpu_status sdrgpu_pipeline_create(sdrgpu_pipeline **out, sdrgpu_channelizer *chan, sdrgpu_bank *bank)
{
    if (!out || !chan || !bank) return fail(SDRGPU_ERR_INVALID_ARG, "NULL argument");
    return sdrgpu_pipeline_create_multi(out, &chan, 1, bank);
}

sdrgpu_status sdrgpu_pipeline_set_chunks(sdrgpu_pipeline *p, int chunks)
{
    if (!p || chunks < 1 || chunks > 64) return fail(SDRGPU_ERR_INVALID_ARG, "chunks must be in [1, 64]");
    p->chunks = chunks;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_pipeline_set_device_chunks(sdrgpu_pipeline *p, int chunks)
{
    if (!p || chunks < 1 || chunks > 64) return fail(SDRGPU_ERR_INVALID_ARG, "chunks must be in [1, 64]");
    p->device_chunks = chunks;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_pipeline_destroy(sdrgpu_pipeline *p)
{
    if (!p) return SDRGPU_OK;
    // the channelizers (and the other banks) were running on the first bank's stream: hand them back their own before
    // that bank (and that stream) can go.  Destroy order: pipeline first, then its channelizers and banks (sdrgpu.h).
    for (auto &e : p->ev_done)
        if (e) {
            cudaEventSynchronize(e);
            cudaEventDestroy(e);
        }
    if (p->copy_in) {
        cudaStreamSynchronize(p->copy_in);
        cudaStreamDestroy(p->copy_in);
    }
    for (auto &s : p->copy_out)
        if (s) {
            cudaStreamSynchronize(s);
            cudaStreamDestroy(s);
        }
    for (cudaEvent_t e : p->copy_events)
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : {p->ev_counts[0], p->ev_counts[1], p->ev_tail, p->ev_h2d})
        if (e) cudaEventDestroy(e);
    for (auto *c : p->chans) sdrgpu_chan_set_stream(c, nullptr);
    for (size_t j = 0; j < p->bank_streams.size(); j++) sdrgpu_bank_set_stream(p->banks[j + 1], p->bank_streams[j]);
    for (auto *d : p->d_rows) cudaFree(d);
    delete p;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_pipeline_process_multi(sdrgpu_pipeline *p, const void *const *iq, int n_floats, int in_mem,
                                            uint8_t *symbols, int symbol_stride, float *demod, long long demod_stride_floats,
                                            int *counts, int out_mem)
{
    if (!p) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    if (p->banks.size() > 1)
        return fail(SDRGPU_ERR_BAD_STATE, "a pipeline of %d banks takes sdrgpu_pipeline_process_routed", (int)p->banks.size());
    const sdrgpu_bank_output out{symbols, symbol_stride, demod, demod_stride_floats, counts};
    return process_sync(p, iq, n_floats, in_mem, &out, out_mem);
}

sdrgpu_status sdrgpu_pipeline_process_routed(sdrgpu_pipeline *p, const void *const *iq, int n_floats, int in_mem,
                                             const sdrgpu_bank_output *outputs, int out_mem)
{
    if (!p || !outputs) return fail(SDRGPU_ERR_INVALID_ARG, "NULL argument");
    return process_sync(p, iq, n_floats, in_mem, outputs, out_mem);
}

sdrgpu_status sdrgpu_pipeline_submit_multi(sdrgpu_pipeline *p, const void *const *iq, int n_floats, uint8_t *symbols,
                                           int symbol_stride, int *counts)
{
    if (!p) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    if (p->banks.size() > 1) return fail(SDRGPU_ERR_BAD_STATE, "asynchronous calls are for one-bank pipelines");
    sdrgpu_bank *b = p->banks[0];
    if (!is_dqpsk(b->cfg.demod)) return fail(SDRGPU_ERR_BAD_STATE, "asynchronous calls are for DQPSK banks (dibits out)");
    if (!symbols || symbol_stride <= 0) return fail(SDRGPU_ERR_INVALID_ARG, "symbols is NULL / symbol_stride <= 0");
    if (p->inflight >= 2) return fail(SDRGPU_ERR_BAD_STATE, "two calls in flight already: sdrgpu_pipeline_wait first");
    const sdrgpu_bank_output out{symbols, symbol_stride, nullptr, 0, counts};
    SDRGPU_TRY(check_call(p, iq, n_floats, &out));
    SDRGPU_CUDA(cudaSetDevice(b->device));
    SDRGPU_TRY(ensure_copy_streams(p));
    // The host buffers go to the device whole, into the staging pair the call in flight does NOT read (the pair used two
    // calls ago: the caller has waited for that call before it could submit this one) -- these copies are what overlaps
    // the other call's kernels -- and the call then runs the device-resident, filters-first schedule on them.
    const int K = (int)p->chans.size();
    std::vector<const void *> staged((size_t)K, nullptr);
    if (n_floats > 0) {
        for (int k = 0; k < K; k++) {
            sdrgpu::chan_swap_staging(p->chans[k]);
            SDRGPU_TRY(sdrgpu::chan_upload(p->chans[k], iq[k], 0, n_floats / 2, p->copy_in));
            staged[(size_t)k] = sdrgpu::chan_staging(p->chans[k]);
        }
        SDRGPU_CUDA(cudaEventRecord(p->ev_h2d, p->copy_in));
        SDRGPU_CUDA(cudaStreamWaitEvent(b->stream, p->ev_h2d, 0));
    }
    bool went_async = false;
    SDRGPU_TRY(process_call(p, staged.data(), n_floats, SDRGPU_DEVICE, &out, SDRGPU_HOST, &went_async));
    // a call that ran to completion (too short to be cut into chunks) is complete when it returns
    if (!went_async) {
        SDRGPU_CUDA(cudaEventRecord(p->ev_counts[p->next_slot], b->stream));
        SDRGPU_CUDA(cudaEventRecord(p->ev_done[p->next_slot], b->stream));
    }
    p->next_slot ^= 1;
    p->inflight++;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_pipeline_wait(sdrgpu_pipeline *p)
{
    if (!p) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    if (p->inflight == 0) return SDRGPU_OK;
    const int oldest = p->inflight == 2 ? p->next_slot : (p->next_slot ^ 1);
    SDRGPU_CUDA(cudaEventSynchronize(p->ev_done[oldest]));
    p->inflight--;
    return SDRGPU_OK;
}

sdrgpu_status sdrgpu_pipeline_process(sdrgpu_pipeline *p, const void *iq, int n_floats, int in_mem, uint8_t *symbols,
                                      int symbol_stride, float *demod, long long demod_stride_floats, int *counts,
                                      int out_mem)
{
    if (!p) return fail(SDRGPU_ERR_INVALID_ARG, "NULL handle");
    if (p->chans.size() != 1) return fail(SDRGPU_ERR_BAD_STATE, "a multi-tuner pipeline takes sdrgpu_pipeline_process_multi");
    if (n_floats > 0 && !iq) return fail(SDRGPU_ERR_INVALID_ARG, "iq is NULL");
    return sdrgpu_pipeline_process_multi(p, &iq, n_floats, in_mem, symbols, symbol_stride, demod, demod_stride_floats, counts,
                                         out_mem);
}

}  // extern "C"
