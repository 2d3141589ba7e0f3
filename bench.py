#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 DSP hot path (contract: see the task's "Measurement" section).

    python bench.py --gpus N --steps K --warmup W [--workload NAME] [--tuners T] [--impl reference] [--no-extra]
                    [--dump-outputs DIR]

Headline workload (default, `c4fm_20m`) = BASELINE.json configs[4]: 20 MS/s tuners -> polyphase channelizer (M = 800)
-> per channel 72-tap FIR -> block AGC -> DQPSK decision-directed timing recovery (P25 Phase 1 C4FM) on all 800 bins,
dibits out.  `--tuners T` tuner streams per GPU feed ONE bank (sdrgpu_pipeline_create_multi): the symbol demodulator is
serial per channel, so it is the number of channels in a launch -- not the length of a buffer -- that fills the GPU.
One "step" = one pass of the chain over one batch of synthetic tuner I/Q: 1 s of every tuner stream of this GPU.
N > 1 is launched by torchrun, one rank per GPU; tuner streams are independent, so every rank processes its own
streams (weak scaling, no data-path collective); torch.distributed is used for the barrier and the max-over-ranks time.

Keys of the JSON line (rank 0): value = whole-job input complex MS/s channelized AND demodulated, inputs resident in
HBM; e2e = the same through the C ABI with pinned HOST buffers (tuner-native 8-bit samples in, dibits out, H2D + D2H
inside the timed region); roofline = the chain against the FP32 ceiling of SURVEY.md 8(d) with the per-kernel table;
cpu_baseline = the oracle (CPU restatement of the reference's Java path) on this box's host cores on a bounded sample;
tuners_per_gpu_curve, configs2_c4fm, configs1_channelizer, configs0_nbfm, configs3_hdqpsk = secondary results (N = 1).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "channelized+demodulated complex MS/s and real-time channel count at 1/2/4/8 GPU"
UNIT = "MS/s"
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # FFMA lanes x 2 flop x max SM clock (SURVEY.md 8d)
DEFAULT_TUNERS = 8                                   # tuner streams per GPU of the headline workload (all of configs[4])

WORKLOADS = {
    # BASELINE.json configs[4]: 20 MS/s tuners -> 800 channels each, full chain (the headline)
    "c4fm_20m": dict(kind="tuner", fs=2e7, taps_per_channel=9, seconds=1.0, demod="c4fm",
                     desc="configs[4]: {t} x 20 MS/s tuner(s) per GPU -> polyphase channelizer (M=800, T=9) -> 72-tap FIR "
                          "+ block AGC + C4FM DQPSK decision-directed timing recovery on all {c} channels, dibits out"),
    # BASELINE.json configs[2]: channelizer + per-channel FIR/AGC + C4FM DQPSK timing recovery on 400 channels
    "c4fm": dict(kind="tuner", fs=1e7, taps_per_channel=9, seconds=1.0, demod="c4fm",
                 desc="configs[2]: {t} x 10 MS/s tuner(s) per GPU -> channelizer (M=400, T=9) + 72-tap FIR + block AGC + "
                      "C4FM DQPSK decision-directed timing recovery on all {c} channels, dibits out"),
    # BASELINE.json configs[1]: polyphase channelizer alone
    "channelizer": dict(kind="tuner", fs=1e7, taps_per_channel=9, seconds=1.0, demod=None,
                        desc="configs[1]: polyphase channelizer 10 MS/s -> 400 x 25 kHz channels (M=400, T=9), "
                             "all bins kept, gain M, [channel][time] output"),
    "channelizer_20m": dict(kind="tuner", fs=2e7, taps_per_channel=9, seconds=1.0, demod=None,
                            desc="configs[4] channelizer stage alone: 20 MS/s -> 800 x 25 kHz channels (M=800, T=9), all "
                                 "bins kept, gain M, [channel][time] output"),
    # BASELINE.json configs[3]: P25 Phase 2 HDQPSK on >= 1000 channel-domain streams
    "hdqpsk_4096": dict(kind="bank", demod="hdqpsk", channels=4096, samples=24 * 1024,
                        desc="configs[3]: P25 Phase 2 HDQPSK, {c} channel-domain streams per GPU at 50 kHz (channel "
                             "samples, not tuner samples): 154-tap FIR + block AGC + Gardner DQPSK timing recovery"),
    # BASELINE.json configs[0] as a many-channel bank: the NBFM chain of NBFMDecoder on channel-domain streams
    "nbfm_4096": dict(kind="bank", demod="nbfm", channels=4096, samples=24 * 1024,
                      desc="configs[0] x {c}: NBFM channel-domain streams per GPU at 50 kHz (channel samples): half-band "
                           "decimate by 2 -> 45-tap FIR -> power squelch -> FM discriminator, 25 kHz floats out"),
}


def workload_config(name, tuners):
    """the `config` object of the JSON line: identical in the GPU arm and the reference arm"""
    cfg = WORKLOADS[name]
    if cfg["kind"] == "tuner":
        m = int(cfg["fs"] / 25000) // 2 * 2
        n_complex = int(cfg["fs"] * cfg["seconds"])
        if cfg["demod"]:
            n_complex = n_complex // (1024 * (m // 2)) * (1024 * (m // 2))
        return {"workload": cfg["desc"].format(t=tuners, c=tuners * m), "tuners_per_gpu": tuners, "channels_per_tuner": m,
                "tuner_rate_hz": cfg["fs"], "channel_rate_hz": 2 * cfg["fs"] / m,
                "input_complex_samples_per_step_per_gpu": tuners * n_complex,
                "l2": "per-step working set (%.0f MB in + %.0f MB channel streams) exceeds the 126 MB L2" %
                      (8 * tuners * n_complex / 1e6, 16.0 * tuners * n_complex / 1e6),
                "sharding": "independent tuner streams per GPU, no collective"}
    c = cfg["channels"]
    return {"workload": cfg["desc"].format(c=c), "channels_per_gpu": c, "samples_per_channel_per_step": cfg["samples"],
            "channel_rate_hz": 50000.0,
            "l2": "per-step working set (%.0f MB in) exceeds the 126 MB L2" % (8.0 * c * cfg["samples"] / 1e6),
            "sharding": "channel rows per GPU, no collective"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(kernel):
    """per-launch DRAM bytes of `kernel` from the committed ncu --set full summary (profiles/traffic.json)"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(kernel)
    except Exception:
        return None


def fir_taps(demod):
    """decoder baseband filters: P25P1DecoderC4FM.java:136-148 (5100/6500 Hz, 72 taps at 50 kHz),
    P25P2DecoderHDQPSK.java:155-166 (6500/7200 Hz, 154 taps), NBFMDecoder.java:306-341 (5000/6250 Hz at 25 kHz, 45 taps)"""
    # designed by the library's host-side restatement of the reference's RemezFIRFilterDesigner (csrc/remez.cpp): the taps
    # the Java decoders run, not another Remez implementation's
    from sdrtrunk_b200.dsp import FilterFactory, FIRFilterSpecification
    spec = {"c4fm": (50000.0, 5100, 6500, 0.01, 0.01, None), "hdqpsk": (50000.0, 6500, 7200, 0.005, 0.01, None),
            "nbfm": (50000.0, 10000, 12500, 0.01, 0.005, True)}.get(demod)
    if spec is None:
        return None
    b = (FIRFilterSpecification.lowPassBuilder().sampleRate(spec[0]).passBandCutoff(spec[1]).passBandAmplitude(1.0)
         .passBandRipple(spec[3]).stopBandAmplitude(0.0).stopBandStart(spec[2]).stopBandRipple(spec[4]))
    if spec[5] is not None:
        b = b.gridDensity(16).oddLength(spec[5])
    taps = FilterFactory.getTaps(b.build())
    assert taps is not None and taps.size == {"c4fm": 72, "hdqpsk": 154, "nbfm": 45}[demod]
    return taps


# ---------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 6:
                self.samples.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
            except ValueError:
                continue
            for name, v in zip(names, s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- CPU baseline
def synth_input_numpy(n_complex, m, seed):
    """bounded CPU-side sample of the synthetic workload: tones on bin centres + AWGN, interleaved float32"""
    rng = np.random.default_rng(seed)
    t = np.arange(n_complex)
    z = 1e-3 * (rng.standard_normal(n_complex) + 1j * rng.standard_normal(n_complex))
    for k in rng.choice(m, 8, replace=False):
        f = (k if k < m // 2 else k - m) / m
        z += 0.05 * np.exp(2j * np.pi * (f * t + rng.uniform()))
    out = np.empty(2 * n_complex, np.float32)
    out[0::2] = z.real
    out[1::2] = z.imag
    return out


class CpuChain:
    """The oracle (kind "port": CPU restatement of the reference Java path; no JVM here) arranged like the
    reference runs it: one channelizer per tuner stream, one output processor + decoder chain per channel.  One
    independent tuner stream (or slice of a bank's channel rows) per host thread (the oracle releases the GIL inside
    its ctypes calls).  The only code in this file that touches oracle/."""

    def __init__(self, workload, threads):
        import oracle
        self.cfg = cfg = WORKLOADS[workload]
        self.workload = workload
        self.threads = threads
        self.states = []
        if cfg["kind"] == "tuner":
            fs = cfg["fs"]
            self.m = m = int(fs / 25000) // 2 * 2
            taps = oracle.sinc_m2_channelizer(fs / m, m, cfg["taps_per_channel"])
            # bounded sample: 1 M input samples, or 2 whole 1024-sample assembler buffers per channel for the chain
            self.n_units = 2 * 1024 * (m // 2) if cfg["demod"] else 1000000
            self.x = synth_input_numpy(self.n_units, m, 1)
            fir = fir_taps(cfg["demod"])
            for _ in range(threads):
                st = {"chan": oracle.Channelizer(taps, m),
                      "procs": [oracle.OneChannelOutputProcessor(50000.0, k, float(m)) for k in range(m)]}
                if cfg["demod"] == "c4fm":
                    st["chains"] = [oracle.P25Chain(oracle.C4FM, 50000.0, fir) for _ in range(m)]
                self.states.append(st)
        else:
            # channel-domain banks: every thread owns `rows` channel rows and runs 4 assembler buffers through each
            self.rows, n = 8, 4 * 1024
            rng = np.random.default_rng(1)
            self.x = (0.3 * rng.standard_normal((self.rows, 2 * n))).astype(np.float32)
            self.n_units = self.rows * n
            fir = fir_taps(cfg["demod"])
            for _ in range(threads):
                if cfg["demod"] == "hdqpsk":
                    st = {"chains": [oracle.P25Chain(oracle.HDQPSK, 50000.0, fir) for _ in range(self.rows)]}
                else:
                    st = {"nbfm": [(oracle.Decimator(2), oracle.ComplexFIR(fir), oracle.SquelchingFMDemodulator(0.0004, -78.0, 4))
                                   for _ in range(self.rows)]}
                self.states.append(st)

    def one_pass(self, st):
        if self.cfg["kind"] == "tuner":
            res = st["chan"].receive(self.x)
            for k in range(self.m):
                # the reference's per-channel extraction (ReusableChannelResultsBuffer.getChannel + gain)
                y = st["procs"][k].process(res)
                if "chains" in st:
                    st["chains"][k].receive(y[: y.size // 2048 * 2048])
        elif "chains" in st:
            for k, chain in enumerate(st["chains"]):
                chain.receive(self.x[k])
        else:
            for k, (dec, fir, fm) in enumerate(st["nbfm"]):
                for b in range(self.x.shape[1] // 2048):      # per 1024-sample assembler buffer, as NBFMDecoder.receive
                    fm.demodulate(fir.filter(dec.decimate_complex(self.x[k, 2048 * b:2048 * (b + 1)])))

    def run(self, reps, threads=None):
        """all threads x reps passes; returns (seconds, units processed): input complex samples (tuner workloads) or
        channel samples (bank workloads)"""
        threads = threads or self.threads
        ths = [threading.Thread(target=lambda s=self.states[i]: [self.one_pass(s) for _ in range(reps)])
               for i in range(threads)]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        return time.perf_counter() - t0, threads * reps * self.n_units

    def describe(self, reps):
        unit = "complex input samples" if self.cfg["kind"] == "tuner" else "channel samples"
        return ("%d threads x %d passes over %d %s each (%s); oracle = C restatement of the reference Java path, JVM "
                "unavailable" % (self.threads, reps, self.n_units, unit, self.workload))


def cpu_baseline(workload, threads, target_seconds=10.0):
    chain = CpuChain(workload, threads)
    chain.run(1, 1)                                   # warm-up
    single_s, n = chain.run(1, 1)
    reps = max(1, int(target_seconds / max(single_s * 1.3, 1e-3)))
    dt, total = chain.run(reps)
    return {"value": total / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
            "single_thread_value": n / single_s / 1e6, "sample": chain.describe(reps)}


# ---------------------------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """Times the reference's CPU implementation of the path (the oracle port; the Java itself cannot run here:
    no JVM) on all host threads, on the GPU arm's workload.  One step = every thread runs `reps` passes over the
    bounded sample."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    chain = CpuChain(args.workload, cores)
    chain.run(1, 1)
    single_s, _ = chain.run(1, 1)
    reps = max(1, int(2.5 / max(single_s * 1.3, 1e-3)))     # ~2.5-3 s per step: thread start / join stays < 1 %
    for _ in range(args.warmup):
        chain.run(reps)
    dt, total = 0.0, 0
    for _ in range(args.steps):
        d, n = chain.run(reps)
        dt += d
        total += n
    value = total / dt / 1e6
    base = {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": chain.describe(reps)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, args.tuners), "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- GPU-side synthetic input
def synth_tones_wideband(torch, dev, m, n_complex, seed):
    """SURVEY.md 8d config 2: one unit-phase-random tone per bin at bin centre + U(-5, 5) kHz, amplitude 1/M each,
    plus AWGN sigma 1e-4 per axis.  Built in the frequency domain (tones on FFT bins of the n_complex-point grid)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    spec = torch.zeros(n_complex, dtype=torch.complex64, device=dev)
    k = torch.arange(m, device=dev)
    centre = torch.where(k < m // 2, k, k - m).double() / m                       # cycles per sample
    off = (torch.rand(m, device=dev, generator=g, dtype=torch.float64) - 0.5) * (10000.0 / (25000.0 * m))
    bins = torch.round((centre + off) * n_complex).long() % n_complex
    ph = 2 * np.pi * torch.rand(m, device=dev, generator=g, dtype=torch.float64)
    spec[bins] = torch.polar(torch.full((m,), float(n_complex) / m, device=dev, dtype=torch.float64), ph).to(torch.complex64)
    z = torch.fft.ifft(spec)
    del spec
    x = torch.view_as_real(z).reshape(-1).contiguous()
    x += 1e-4 * torch.randn(x.shape, device=dev, generator=g, dtype=torch.float32)
    return x


def synth_c4fm_wideband(torch, dev, m, n_ch, seed, amplitude=0.02, noise=2e-3):
    """SURVEY.md 8d config 3: every bin carries a continuous C4FM stream (4800 sym/s, deviation levels +/-1, +/-3 ->
    phase steps of level * pi/4 per symbol, raised-cosine frequency pulses), random dibits, carrier offset U(-200, 200)
    Hz and timing phase per channel; channels are multiplexed onto the bin centres in the frequency domain."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    fs_ch, sym_rate = 50000.0, 4800.0
    sps = fs_ch / sym_rate
    n_sym = int(n_ch / sps) + 8
    dibits = torch.randint(0, 4, (m, n_sym), device=dev, generator=g)
    levels = torch.tensor([1.0, 3.0, -1.0, -3.0], device=dev, dtype=torch.float64)[dibits]
    off = (torch.rand(m, 1, device=dev, generator=g, dtype=torch.float64) - 0.5) * 400.0
    tphase = torch.rand(m, 1, device=dev, generator=g, dtype=torch.float64)
    phase0 = 2 * np.pi * torch.rand(m, 1, device=dev, generator=g, dtype=torch.float64)
    n = torch.arange(n_ch, device=dev, dtype=torch.float64).unsqueeze(0)
    n_w = n_ch * m // 2
    spec = torch.zeros(n_w, dtype=torch.complex64, device=dev)
    quarter = n_ch // 4
    j = torch.cat([torch.arange(0, quarter, device=dev), torch.arange(-quarter, 0, device=dev)])
    for lo in range(0, m, 50):                       # 50 channels at a time bounds the float64 temporaries
        hi = min(m, lo + 50)
        t = n / sps - tphase[lo:hi]
        k = torch.floor(t).long()
        valid = (k >= 0) & (k < n_sym)
        u = t - k - 0.5
        pulse = 1.0 + torch.cos(2 * np.pi * u)
        lv = torch.gather(levels[lo:hi], 1, k.clamp(0, n_sym - 1))
        freq = torch.where(valid, lv * pulse, torch.zeros_like(pulse))
        phase = torch.cumsum(freq, dim=1) * (np.pi / 4.0) / sps + 2 * np.pi * off[lo:hi] * n / fs_ch + phase0[lo:hi]
        xf = torch.fft.fft(torch.polar(torch.full_like(phase, amplitude), phase).to(torch.complex64), dim=1)
        for c in range(lo, hi):
            centre = (c if c < m // 2 else c - m) * (n_ch // 2)
            spec[(centre + j) % n_w] += xf[c - lo, j % n_ch]
        del t, k, valid, u, pulse, lv, freq, phase, xf
    z = torch.fft.ifft(spec) * (n_w / n_ch)
    del spec
    x = torch.view_as_real(z).reshape(-1).contiguous()
    x += noise * torch.randn(x.shape, device=dev, generator=g, dtype=torch.float32)
    return x, dibits.to(torch.uint8).cpu().numpy()


def dibit_match(decoded, truth, skip=300):
    """fraction of decoded dibits equal to the transmitted ones after acquisition, best over small lags"""
    best = 0.0
    for lag in range(0, 24):
        n = min(decoded.size - lag, truth.size) - 20
        if n > skip + 100:
            best = max(best, float(np.mean(decoded[lag + skip:lag + n] == truth[skip:n])))
    return best


def valid_prefix(buf, counts):
    """rows of `buf` with everything past each row's count zeroed: a caller reads only the first count values, so what
    a step leaves behind them is not part of its output"""
    out = buf.copy()
    out[np.arange(buf.shape[1])[None, :] >= counts[:, None]] = 0
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """writes every array as DIR/<name>.npy in float32.  Arrays of up to 1 MB are written whole; the larger ones share
    the rest of DUMP_LIMIT_BYTES and keep a fixed, seeded sample of their rows when they do not fit, listed in
    DIR/<name>_rows.npy (the same rows on every run, so that the dumps of two builds compare value for value)."""
    os.makedirs(directory, exist_ok=True)
    small = {k for k, a in arrays.items() if a.size * 4 <= 1 << 20}
    room = DUMP_LIMIT_BYTES - sum(arrays[k].size * 4 for k in small) - (1 << 20)   # 1 MB for row lists and headers
    large = sum(a.size * 4 for k, a in arrays.items() if k not in small)
    for name, a in sorted(arrays.items()):
        if name not in small and large > room:
            keep = max(1, int(a.shape[0] * room / large))
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))
            np.save(os.path.join(directory, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def synth_dqpsk_channels(torch, dev, n_channels, n, seed, symbol_rate=6000.0, fs=50000.0, beta=0.35, noise=0.03):
    """SURVEY.md 8d config 4: channel-domain pi/4-DQPSK streams (raised-cosine shaped impulse train evaluated at the
    non-integer 8.33 samples per symbol), carrier offset U(-200, 200) Hz and timing phase per channel, + AWGN."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    sps = fs / symbol_rate
    n_sym = int(n / sps) + 16
    out = torch.empty((n_channels, 2 * n), dtype=torch.float32, device=dev)
    truth = torch.empty((n_channels, n_sym), dtype=torch.uint8)
    levels = torch.tensor([1.0, 3.0, -1.0, -3.0], device=dev, dtype=torch.float64)
    idx = torch.arange(n, device=dev, dtype=torch.float64).unsqueeze(0)
    for lo in range(0, n_channels, 256):
        hi = min(n_channels, lo + 256)
        c = hi - lo
        dib = torch.randint(0, 4, (c, n_sym), device=dev, generator=g)
        truth[lo:hi] = dib.to(torch.uint8).cpu()
        sym = torch.polar(torch.ones((c, n_sym), device=dev, dtype=torch.float64),
                          torch.cumsum(levels[dib] * (np.pi / 4.0), dim=1))
        off = (torch.rand(c, 1, device=dev, generator=g, dtype=torch.float64) - 0.5) * 400.0
        tph = torch.rand(c, 1, device=dev, generator=g, dtype=torch.float64)
        t = idx / sps - tph
        k0 = torch.floor(t).long()
        z = torch.zeros((c, n), dtype=torch.complex128, device=dev)
        for dk in range(-6, 8):
            k = k0 + dk
            valid = (k >= 0) & (k < n_sym)
            u = t - k
            den = 1.0 - (2 * beta * u) ** 2
            pulse = torch.where(den.abs() < 1e-9, torch.full_like(u, (np.pi / 4) * np.sinc(1 / (2 * beta))),
                                torch.sinc(u) * torch.cos(np.pi * beta * u) / den)
            z += torch.where(valid, torch.gather(sym, 1, k.clamp(0, n_sym - 1)) * pulse, torch.zeros_like(z))
        z = z * torch.polar(torch.ones_like(idx), 2 * np.pi * off * idx / fs)
        zr = torch.view_as_real(z.to(torch.complex64)).reshape(c, 2 * n)
        out[lo:hi] = zr + noise * torch.randn(zr.shape, device=dev, generator=g, dtype=torch.float32)
        del sym, t, k0, z, zr
    return out, truth.numpy()


def synth_nbfm_channels(torch, dev, n_channels, n, seed, fs=50000.0, noise=3e-5):
    """configs[0] as a bank: channel-domain NBFM carriers at 50 kHz (audio tone 300-3000 Hz, +/-2.5 kHz deviation,
    amplitude 0.5, carrier offset U(-500, 500) Hz) + AWGN; every 8th channel carries noise only (stays squelched)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    out = torch.empty((n_channels, 2 * n), dtype=torch.float32, device=dev)
    t = torch.arange(n, device=dev, dtype=torch.float64).unsqueeze(0) / fs
    for lo in range(0, n_channels, 512):
        hi = min(n_channels, lo + 512)
        c = hi - lo
        audio = 300.0 + 2700.0 * torch.rand(c, 1, device=dev, generator=g, dtype=torch.float64)
        off = (torch.rand(c, 1, device=dev, generator=g, dtype=torch.float64) - 0.5) * 1000.0
        phase = (2500.0 / audio) * torch.sin(2 * np.pi * audio * t) + 2 * np.pi * off * t
        amp = torch.full((c, 1), 0.5, device=dev, dtype=torch.float64)
        amp[(torch.arange(lo, hi, device=dev) % 8) == 7] = 0.0
        z = torch.polar(amp.expand(c, n).contiguous(), phase).to(torch.complex64)
        zr = torch.view_as_real(z).reshape(c, 2 * n)
        out[lo:hi] = zr + noise * torch.randn(zr.shape, device=dev, generator=g, dtype=torch.float32)
        del phase, z, zr
    return out


# ---------------------------------------------------------------------------------------------- GPU arm
def make_timed(torch, dist, dev, world):
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, stream, steps, warmup):
        """W untimed + K timed steps: CUDA events on the launching stream, barrier + synchronize on both sides, max over
        ranks; also the wall clock of the K steps (what a caller of the blocking host-buffer API sees)"""
        for _ in range(warmup):
            fn()
        barrier()
        start = torch.cuda.Event(enable_timing=True)
        stop = torch.cuda.Event(enable_timing=True)
        start.record(stream)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        stop.record(stream)
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        ms = start.elapsed_time(stop)
        if world > 1:
            tt = torch.tensor([ms, wall], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms, wall = tt.tolist()
        return ms, wall

    return barrier, timed


class TunerInputs:
    """synthetic tuner streams of one workload shape, generated once on the device and shared by the workloads of
    different tuner counts (the first T streams)"""

    def __init__(self, torch, dev, name, rank, count):
        cfg = WORKLOADS[name]
        fs = cfg["fs"]
        self.m = m = int(fs / 25000) // 2 * 2
        n_complex = int(fs * cfg["seconds"])
        if cfg["demod"]:
            n_complex = n_complex // (1024 * (m // 2)) * (1024 * (m // 2))    # whole assembler buffers
        self.n_complex, self.n_blocks = n_complex, n_complex // (m // 2)
        self.x, self.truth = [], []
        for k in range(count):
            if cfg["demod"] == "c4fm":
                x, truth = synth_c4fm_wideband(torch, dev, m, self.n_blocks, seed=3 + 1000 * rank + 17 * k, amplitude=8.0 / m)
            else:
                x, truth = synth_tones_wideband(torch, dev, m, n_complex, seed=2 + 1000 * rank + 17 * k), None
            self.x.append(x)
            self.truth.append(truth)


class TunerWorkload:
    """T tuner streams of one GPU: T channelizers (+ one bank over all their channels + the multi-tuner pipeline)."""

    def __init__(self, name, inputs, tuners, local_rank, bins=None):
        import torch
        from sdrtrunk_b200 import native
        from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline
        self.torch, self.native, self.L = torch, native, native.lib()
        self.name, self.cfg, self.T = name, WORKLOADS[name], tuners
        cfg = self.cfg
        fs = cfg["fs"]
        self.m = m = inputs.m
        self.n_complex, self.n_blocks = inputs.n_complex, inputs.n_blocks     # per tuner
        self.n_floats = 2 * self.n_complex
        self.total_complex = tuners * self.n_complex
        self.dev = dev = torch.device("cuda", local_rank)
        self.x_dev = inputs.x[:tuners]
        self.truth = inputs.truth[:tuners]
        self.stream = torch.cuda.Stream(device=dev)
        self.chans = []
        # level 2 of SURVEY.md 8e: this rank keeps (and demodulates) the polyphase bins [lo, hi) of every tuner
        self.bins = bins if bins is not None else (0, m)
        self.rows_per_tuner = self.bins[1] - self.bins[0]
        for _ in range(tuners):
            ch = ComplexPolyphaseChannelizerM2(fs, cfg["taps_per_channel"], device=local_rank, maxInputFloats=self.n_floats)
            if bins is not None:
                ch.setChannels(list(range(*bins)))
            ch.setStream(self.stream.cuda_stream)
            self.chans.append(ch)
        self.pipeline = None
        self._host = {}
        self.fmt = "f32"
        if cfg["demod"]:
            rows = tuners * self.rows_per_tuner
            self.bank = Bank.preset(native.PRESET_P25_C4FM, rows, 2 * fs / m, fir_taps("c4fm"),
                                    max_samples_per_call=self.n_blocks, device=local_rank)
            self.bank.setStream(self.stream.cuda_stream)
            self.pipeline = Pipeline(self.chans, self.bank)
            self.chunks = int(os.environ.get("SDRGPU_BENCH_CHUNKS", "8"))
            self.device_chunks = int(os.environ.get("SDRGPU_BENCH_DEVICE_CHUNKS", "1" if tuners == 1 else "6"))
            self.pipeline.setChunks(self.chunks)
            self.pipeline.setDeviceChunks(self.device_chunks)
            self.sym_stride = self.n_blocks // 8 + 64          # > 4800/50000 symbols per sample
            self.sym_dev = torch.zeros((rows, self.sym_stride), dtype=torch.uint8, device=dev)
            self.cnt_dev = torch.zeros(rows, dtype=torch.int32, device=dev)
            self.sym_host = torch.zeros((rows, self.sym_stride), dtype=torch.uint8, pin_memory=True)
            self.cnt_host = torch.zeros(rows, dtype=torch.int32, pin_memory=True)
            self.d2h = self.sym_host.numel() + 4 * rows
        else:
            assert tuners == 1
            self.out_dev = torch.empty((m, 2 * self.n_blocks), dtype=torch.float32, device=dev)
            self.out_host = torch.empty((m, 2 * self.n_blocks), dtype=torch.float32, pin_memory=True)
            self.d2h = self.out_host.numel() * 4
        self._dev_ptrs = (C.c_void_p * tuners)(*[x.data_ptr() for x in self.x_dev])

    # ---- input formats of the host-buffer path
    def host_inputs(self, fmt):
        """pinned host copies of the tuner streams in a tuner's native sample format (converted on the device)"""
        torch = self.torch
        if fmt not in self._host:
            bufs = []
            for x in self.x_dev:
                if fmt == "f32":
                    h = torch.empty(self.n_floats, dtype=torch.float32, pin_memory=True)
                    h.copy_(x)
                elif fmt == "s8":      # SignedByteSampleConverter: x / 128
                    h = torch.empty(self.n_floats, dtype=torch.int8, pin_memory=True)
                    h.copy_(torch.clamp(torch.round(x * 128.0), -128, 127).to(torch.int8))
                elif fmt == "u8":      # ByteSampleConverter: (x - 127) / 128
                    h = torch.empty(self.n_floats, dtype=torch.uint8, pin_memory=True)
                    h.copy_(torch.clamp(torch.round(x * 128.0 + 127.0), 0, 255).to(torch.uint8))
                else:
                    raise ValueError(fmt)
                bufs.append(h)
            self._host[fmt] = (bufs, (C.c_void_p * self.T)(*[h.data_ptr() for h in bufs]))
        return self._host[fmt]

    def set_format(self, fmt):
        if fmt != self.fmt:
            for ch in self.chans:
                ch.setSampleFormat(fmt)
            self.fmt = fmt

    def bytes_per_value(self, fmt):
        return {"f32": 4, "s8": 1, "u8": 1}[fmt]

    def step_device(self):
        n, L = self.native, self.L
        if self.pipeline is None:
            n.check(L.sdrgpu_chan_process(self.chans[0]._h, self._dev_ptrs[0], self.n_floats, n.DEVICE,
                                          C.c_void_p(self.out_dev.data_ptr()), 2 * self.n_blocks, n.DEVICE,
                                          n.LAYOUT_CHANNELS, None))
        else:
            n.check(L.sdrgpu_pipeline_process_multi(self.pipeline._h, self._dev_ptrs, self.n_floats, n.DEVICE,
                                                    C.c_void_p(self.sym_dev.data_ptr()), self.sym_stride, None, 0,
                                                    C.c_void_p(self.cnt_dev.data_ptr()), n.DEVICE))

    def step_host(self):
        n, L = self.native, self.L
        _, ptrs = self.host_inputs(self.fmt)
        if self.pipeline is None:
            n.check(L.sdrgpu_chan_process(self.chans[0]._h, ptrs[0], self.n_floats, n.HOST,
                                          C.c_void_p(self.out_host.data_ptr()), 2 * self.n_blocks, n.HOST,
                                          n.LAYOUT_CHANNELS, None))
        else:
            n.check(L.sdrgpu_pipeline_process_multi(self.pipeline._h, ptrs, self.n_floats, n.HOST,
                                                    C.c_void_p(self.sym_host.data_ptr()), self.sym_stride, None, 0,
                                                    C.c_void_p(self.cnt_host.data_ptr()), n.HOST))

    def step_host_stream(self):
        """the host-buffer step as a continuous stream delivers it: sdrgpu_pipeline_submit_multi with two calls in flight
        (the H2D copies of step k + 1 overlap the kernels of step k), alternating pinned output buffers; every step still
        copies its whole input in and its dibits + counts out"""
        n, L = self.native, self.L
        _, ptrs = self.host_inputs(self.fmt)
        if not hasattr(self, "_stream_out"):
            torch = self.torch
            self._stream_out = [(self.sym_host, self.cnt_host),
                                (torch.zeros_like(self.sym_host).pin_memory(), torch.zeros_like(self.cnt_host).pin_memory())]
            self._stream_k, self._stream_inflight = 0, 0
        sym, cnt = self._stream_out[self._stream_k & 1]
        n.check(L.sdrgpu_pipeline_submit_multi(self.pipeline._h, ptrs, self.n_floats, C.c_void_p(sym.data_ptr()),
                                               self.sym_stride, C.c_void_p(cnt.data_ptr())))
        self._stream_k += 1
        self._stream_inflight += 1
        if self._stream_inflight == 2:
            n.check(L.sdrgpu_pipeline_wait(self.pipeline._h))
            self._stream_inflight -= 1

    def stream_drain(self):
        while getattr(self, "_stream_inflight", 0) > 0:
            self.native.check(self.L.sdrgpu_pipeline_wait(self.pipeline._h))
            self._stream_inflight -= 1

    def outputs(self):
        """what the last device-resident step handed its caller: the dibits of every channel row (zero past the row's
        count) and the counts, or the channelizer's [channel][time] streams"""
        if self.pipeline is None:
            return {"channels": self.out_dev.cpu().numpy()}
        cnt = self.cnt_dev.cpu().numpy()
        return {"dibits": valid_prefix(self.sym_dev.cpu().numpy(), cnt), "dibit_counts": cnt}

    def sanity(self):
        """decoded-vs-transmitted dibits of a few rows (first pass over the streams, from the reset state; a plausibility
        figure for the timed workload -- parity itself is tests/)"""
        if self.pipeline is None or self.truth[0] is None:
            return None
        self.set_format("f32")
        self.host_inputs("f32")
        self.step_host()
        cnt = self.cnt_host.numpy()
        out = {}
        per = self.rows_per_tuner
        rows = self.T * per
        for r in sorted({0, min(57, per - 1), per // 2, per - 1, rows - per + min(3, per - 1), rows - 1}):
            t, c = divmod(r, per)
            dec = self.sym_host.numpy()[r, :cnt[r]]
            out["tuner%d_bin%d" % (t, self.bins[0] + c)] = {
                "symbols": int(cnt[r]), "match_after_acquisition": round(dibit_match(dec, self.truth[t][self.bins[0] + c]), 4)}
        if self.T > 1 or self.n_floats > 50000000:
            self._host.pop("f32", None)        # hundreds of MB of pinned memory per tuner: only kept for T = 1
        return out

    def kernel_times(self, steps):
        """per-kernel device time, live, CUDA events on the launching stream (own loop so that the per-step event
        synchronisation does not perturb the throughput numbers): one full-size launch per kernel"""
        for ch in self.chans:
            ch.enableTiming(True)
        if self.pipeline is not None:
            self.bank.enableTiming(True)
            self.pipeline.setDeviceChunks(1)
        rows = []
        self.set_format("f32")
        for _ in range(steps):
            self.step_device()
            row = {"pfb_ifft": sum(ch.lastKernelMs() for ch in self.chans)}
            if self.pipeline is not None:
                f, d = self.bank.lastKernelMs()
                row.update({"fir_agc": f, "psk": d})
            rows.append(row)
        for ch in self.chans:
            ch.enableTiming(False)
        if self.pipeline is not None:
            self.bank.enableTiming(False)
            self.pipeline.setDeviceChunks(self.device_chunks)
        return {k: statistics.mean(r[k] for r in rows) for k in rows[0]}

    def dispose(self):
        if self.pipeline is not None:
            self.pipeline.dispose()
            self.bank.dispose()
        for ch in self.chans:
            ch.dispose()


def measure_tuner(w, args, world, timed, full=True, capture=False):
    """device-resident and host-buffer throughput of one TunerWorkload; `full` adds the secondary variants, `capture`
    keeps the outputs of the last timed device-resident step (res["outputs"])"""
    L = w.L
    steps = args.steps
    sanity = w.sanity() if (full and not args.device_only) else None
    w.set_format("f32")
    launches0 = L.sdrgpu_launch_count()
    ms_dev, _ = timed(w.step_device, w.stream, steps, args.warmup)
    launches = (L.sdrgpu_launch_count() - launches0) * steps // (steps + args.warmup)
    total = w.total_complex * world
    res = {"ms_per_step": ms_dev / steps, "value": total / (ms_dev / steps * 1e-3) / 1e6, "launches": launches,
           "sanity": sanity}
    if capture:
        res["outputs"] = w.outputs()        # before the legs below run the same buffers again

    def e2e_leg(fmt, note):
        w.set_format(fmt)
        w.host_inputs(fmt)
        ms, wall = timed(w.step_host, w.stream, steps, max(3, args.warmup))
        per = max(ms, wall) / steps       # the blocking call: device time of the stream and the caller's wall clock
        return {"value": total / (per * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": w.T * w.n_floats * w.bytes_per_value(fmt),
                "d2h_bytes_per_step": w.d2h, "ms_per_step": per, "input": note}

    def e2e_stream_leg(fmt, note):
        # K steps with two calls in flight; the timed region ends with a full device synchronise (wall clock), which is
        # when the last step's dibits are on the host
        w.set_format(fmt)
        w.host_inputs(fmt)
        ms, wall = timed(w.step_host_stream, w.stream, steps, max(3, args.warmup))
        w.stream_drain()
        per = max(ms, wall) / steps
        return {"value": total / (per * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": w.T * w.n_floats * w.bytes_per_value(fmt),
                "d2h_bytes_per_step": w.d2h, "ms_per_step": per, "input": note}

    if not args.device_only:
        if w.pipeline is not None:
            # the chain's host-buffer path takes what a 20 MS/s USB tuner delivers: signed 8-bit I/Q (HackRF;
            # SignedByteSampleConverter), converted on the device in front of the channelizer
            note = ("tuner-native signed 8-bit I/Q in pinned host buffers (SignedByteSampleConverter format, converted on the "
                    "device), dibits + counts back to pinned host buffers; ")
            blocking = e2e_leg("s8", note + "one blocking sdrgpu_pipeline_process_multi call per step")
            stream = e2e_stream_leg("s8", note + "a continuous stream: sdrgpu_pipeline_submit_multi / _wait with two steps in "
                                                 "flight, every step's H2D and D2H copies inside the timed region")
            # the host side picks the call that suits its bank: the stream wins once the bank fills the GPU, a single tuner's
            # latency-bound step is served better by the chunked blocking call
            res["e2e"] = dict(stream if stream["value"] >= blocking["value"] else blocking)
            res["e2e"]["stream_two_in_flight"] = {"value": stream["value"], "unit": UNIT, "ms_per_step": stream["ms_per_step"]}
            res["e2e"]["blocking_call"] = {"value": blocking["value"], "unit": UNIT, "ms_per_step": blocking["ms_per_step"]}
            if full and w.T == 1:
                res["e2e_f32_input"] = e2e_leg("f32", "float32 I/Q in pinned host buffers (the reference's float[] buffers)")
        else:
            res["e2e"] = e2e_leg("f32", "float32 I/Q in pinned host buffers, [channel][time] float32 streams back")
            if full:
                res["e2e_u8_input"] = e2e_leg("u8", "unsigned 8-bit tuner samples (ByteSampleConverter format), converted on "
                                                    "the device")
        w.set_format("f32")
    res["kernels"] = w.kernel_times(min(steps, 10))
    if full and w.pipeline is not None:
        # section 8f #3: the same step with the P25 Phase 1 sync detector + PLL inversion feedback running in the
        # demodulator kernel
        w.bank.setSyncDetector(w.native.SYNC_P25_PHASE1)
        ms_sync, _ = timed(w.step_device, w.stream, steps, 3)
        w.bank.setSyncDetector(w.native.SYNC_NONE)
        res["with_sync"] = {"ms_per_step": ms_sync / steps, "value": total / (ms_sync / steps * 1e-3) / 1e6, "unit": UNIT}
    if full and w.pipeline is not None:
        # the usual sdrtrunk situation: every channel frequency-corrected (OneChannelOutputProcessor + Oscillator);
        # small offsets so that the demodulators keep their locks on the synthetic channels.  Measured last: the
        # selection change restarts the channel oscillators.  The oscillator look-ahead runs on a side stream: the
        # wall clock of the loop with a full device synchronise is reported beside the stream's event time.
        for ch in w.chans:
            ch.setOutputChannels([([k], 37 if k % 2 else -53) for k in range(w.m)])
        ms_corr, wall_corr = timed(w.step_device, w.stream, steps, 3)
        res["corrected"] = {"ms_per_step": ms_corr / steps, "wall_ms_per_step_with_device_sync": wall_corr / steps,
                            "value": total / (ms_corr / steps * 1e-3) / 1e6, "unit": UNIT}
    if full and w.pipeline is None:
        res["airspy"] = measure_airspy(w, args, world, timed)
    return res


def measure_airspy(w, args, world, timed):
    """section 8f #1: Airspy native buffers (packed 12-bit real samples at twice the complex rate, 3 bytes per complex
    sample), unpacked + DC-removed + Hilbert-transformed on the device (AirspySampleConverter).  Random ADC codes: this
    leg measures throughput, parity is tests/."""
    torch, n, L = w.torch, w.native, w.L
    g = torch.Generator(device=w.dev)
    g.manual_seed(77)
    nbytes = w.n_floats // 2 * 3
    x_dev = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device=w.dev, generator=g)
    x_host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    x_host.copy_(x_dev)
    w.chans[0].setSampleFormat("airspy_packed")

    def dev_step():
        n.check(L.sdrgpu_chan_process(w.chans[0]._h, C.c_void_p(x_dev.data_ptr()), w.n_floats, n.DEVICE,
                                      C.c_void_p(w.out_dev.data_ptr()), 2 * w.n_blocks, n.DEVICE, n.LAYOUT_CHANNELS, None))

    def host_step():
        n.check(L.sdrgpu_chan_process(w.chans[0]._h, C.c_void_p(x_host.data_ptr()), w.n_floats, n.HOST,
                                      C.c_void_p(w.out_host.data_ptr()), 2 * w.n_blocks, n.HOST, n.LAYOUT_CHANNELS, None))

    ms_a, _ = timed(dev_step, w.stream, args.steps, 3)
    out = {"input": "Airspy packed 12-bit real samples (3 bytes per complex sample): unpack + DC removal + Hilbert "
                    "transform on the device in front of the channelizer",
           "device_resident": {"ms_per_step": ms_a / args.steps,
                               "value": w.n_complex * world / (ms_a / args.steps * 1e-3) / 1e6, "unit": UNIT}}
    if not args.device_only:
        ms_h, wall_h = timed(host_step, w.stream, args.steps, 3)
        a_ms = max(ms_h, wall_h) / args.steps
        out["e2e"] = {"value": w.n_complex * world / (a_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": a_ms,
                      "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": w.d2h}
    w.chans[0].setSampleFormat("f32")
    w.fmt = "f32"
    return out


def chain_flop_per_input_sample(m, n_fir):
    """SURVEY.md 8(d): filter bank 4 T 2 + FFT 5 log2(M) 2 + 2 channel samples x (4 N_fir + ~40)"""
    return 72.0 + 10.0 * np.log2(m) + 2.0 * (4.0 * n_fir + 40.0)


def roofline_tuner(w, r, peak, peak_src, steps):
    """chain workloads: FP32 ceiling of SURVEY.md 8(d) for the whole step + the per-kernel table; channelizer alone: HBM"""
    k = r["kernels"]
    alg_hbm = 24.0 * w.total_complex      # 8 B read + 16 B written per input complex sample, all M bins kept
    pfb = {"kernel": "pfb2_kernel", "bound": "hbm", "ms": k["pfb_ifft"], "launches_per_step": w.T,
           "achieved": alg_hbm / (k["pfb_ifft"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
           "frac": alg_hbm / (k["pfb_ifft"] * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_step": alg_hbm}
    if w.pipeline is None:
        # a step of this workload is exactly one launch of the kernel, so its average launch duration over the timed
        # region is the step time; the per-launch time with a synchronisation after every step is reported beside it
        single = r["launches"] == steps
        k_ms = r["ms_per_step"] if single else k["pfb_ifft"]
        ach = alg_hbm / (k_ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": load_traffic("pfb2_kernel_m%d" % w.m), "kernel": "pfb2_kernel", "kernel_ms": k_ms,
                "kernel_ms_isolated": k["pfb_ifft"], "algorithmic_bytes_per_launch": alg_hbm, "peak_source": peak_src}
    n_ch = 2.0 * w.total_complex           # channel samples per step (2x oversampled)
    n_fir = 72
    fir_flop, psk_flop = n_ch * 4.0 * n_fir, n_ch * 40.0
    chain_flop = chain_flop_per_input_sample(w.m, n_fir) * w.total_complex
    ach = chain_flop / (r["ms_per_step"] * 1e-3) / 1e12
    table = [pfb,
             {"kernel": "fir_agc_split_kernel", "bound": "fp32", "ms": k["fir_agc"], "launches_per_step": 1,
              "achieved": fir_flop / (k["fir_agc"] * 1e-3) / 1e12, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s",
              "frac": fir_flop / (k["fir_agc"] * 1e-3) / 1e12 / FP32_PEAK_TFLOPS, "algorithmic_flop_per_step": fir_flop},
             {"kernel": "psk_multi_kernel", "bound": "latency (serial per-symbol feedback loop); fp32 view", "ms": k["psk"],
              "launches_per_step": 1, "achieved": psk_flop / (k["psk"] * 1e-3) / 1e12, "peak": FP32_PEAK_TFLOPS,
              "unit": "TFLOP/s", "frac": psk_flop / (k["psk"] * 1e-3) / 1e12 / FP32_PEAK_TFLOPS,
              "algorithmic_flop_per_step": psk_flop,
              "channels_in_launch": w.T * w.m}]
    return {"bound": "fp32", "achieved": ach, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": ach / FP32_PEAK_TFLOPS,
            "traffic": load_traffic("chain_%s_t%d" % (w.name, w.T)),
            "kernel": "chain: pfb2_kernel x %d + fir_agc_split_kernel + psk_multi_kernel (whole step; the demodulator overlaps the "
                      "filters of the next time chunk)" % w.T,
            "kernel_ms": r["ms_per_step"], "algorithmic_flop_per_input_sample": chain_flop_per_input_sample(w.m, n_fir),
            "algorithmic_flop_per_step": chain_flop, "peak_source": "148 SM x 128 FFMA lanes x 2 x 1.965 GHz (SURVEY.md 8d)",
            "hbm_peak_source": peak_src, "kernels": table}


def realtime_channels(value_msps, world, m, fs):
    """channels x achieved rate / required rate: how many 25 kHz channels this throughput serves in real time"""
    return m * value_msps / (fs / 1e6)


def summarize_tuner(w, r, peak, peak_src, steps, world):
    """secondary-result object of one measured TunerWorkload"""
    out = {"workload": workload_config(w.name, w.T)["workload"], "tuners_per_gpu": w.T, "value": r["value"], "unit": UNIT,
           "ms_per_step": r["ms_per_step"], "realtime_channels": realtime_channels(r["value"], world, w.m, w.cfg["fs"]),
           "gpu_launches": r["launches"], "kernels_ms": r["kernels"], "roofline": roofline_tuner(w, r, peak, peak_src, steps)}
    for key, name in (("e2e", "e2e"), ("e2e_f32_input", "e2e_f32_input"), ("e2e_u8_input", "e2e_u8_input"),
                      ("with_sync", "with_sync_detector"), ("corrected", "with_frequency_corrected_channels"),
                      ("airspy", "airspy_input"), ("sanity", "decode_sanity")):
        if r.get(key) is not None:
            out[name] = r[key]
    return out


# ---------------------------------------------------------------------------------------------- channel-domain banks
def run_bank(name, args, rank, world, local_rank, torch, dist, as_secondary=False):
    """BASELINE configs[3] (hdqpsk_4096: 154-tap FIR -> AGC -> Gardner timing recovery) and configs[0] as a bank
    (nbfm_4096: decimate by 2 -> 45-tap FIR -> squelching FM discriminator) on channel-domain streams, no channelizer.
    Channels are sharded over the ranks (level 3 of SURVEY 8e)."""
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import Bank
    L = native.lib()
    cfg = WORKLOADS[name]
    dev = torch.device("cuda", local_rank)
    barrier, timed = make_timed(torch, dist, dev, world)
    channels = int(os.environ.get("SDRGPU_BENCH_CHANNELS", str(cfg["channels"])))
    n = cfg["samples"]                                             # 0.49 s of signal per step
    fir = fir_taps(cfg["demod"])
    hd = cfg["demod"] == "hdqpsk"
    if hd:
        x, truth = synth_dqpsk_channels(torch, dev, channels, n, seed=4 + 1000 * rank)
        bank = Bank.preset(native.PRESET_P25_HDQPSK, channels, 50000.0, fir, max_samples_per_call=n, device=local_rank)
    else:
        x, truth = synth_nbfm_channels(torch, dev, channels, n, seed=5 + 1000 * rank), None
        bank = Bank.preset(native.PRESET_NBFM, channels, 50000.0, fir, max_samples_per_call=n, device=local_rank)
    stream = torch.cuda.Stream(device=dev)
    bank.setStream(stream.cuda_stream)
    if hd:
        stride = n // 7 + 64
        sym = torch.zeros((channels, stride), dtype=torch.uint8, device=dev)
        sym_host = torch.zeros((channels, stride), dtype=torch.uint8, pin_memory=True)
        dem, dem_host, dstride = None, None, 0
    else:
        stride, sym, sym_host = 0, None, None
        dstride = n // 2
        dem = torch.zeros((channels, dstride), dtype=torch.float32, device=dev)
        dem_host = torch.zeros((channels, dstride), dtype=torch.float32, pin_memory=True)
    cnt = torch.zeros(channels, dtype=torch.int32, device=dev)
    cnt_host = torch.zeros(channels, dtype=torch.int32, pin_memory=True)
    x_host = torch.empty(x.shape, dtype=torch.float32, pin_memory=True)
    x_host.copy_(x)
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None

    def step():
        native.check(L.sdrgpu_bank_process(bank._h, vp(x), 2 * n, n, native.DEVICE, vp(sym), stride, vp(dem), dstride,
                                           vp(cnt), native.DEVICE))

    def step_host():
        native.check(L.sdrgpu_bank_process(bank._h, vp(x_host), 2 * n, n, native.HOST, vp(sym_host), stride, vp(dem_host),
                                           dstride, vp(cnt_host), native.HOST))

    step()
    barrier()
    sanity = None
    if hd:
        first, counts = sym.cpu().numpy(), cnt.cpu().numpy()
        sanity = {str(c): round(dibit_match(first[c, :counts[c]], truth[c], skip=300), 4) for c in (0, channels // 4, channels - 1)}
    else:
        d = dem.cpu().numpy()
        # open channels carry the audio tone at +/-2.5 kHz deviation: peak angle 2 pi 2500 / 25000; squelched ones are 0
        sanity = {"open_channel_peak": round(float(np.max(np.abs(d[0, 2000:]))), 4),
                  "expected_peak": round(2 * np.pi * 2500 / 25000, 4),
                  "squelched_channel_peak": float(np.max(np.abs(d[7])))}
    launches0 = L.sdrgpu_launch_count()
    ms, _ = timed(step, stream, args.steps, args.warmup)
    launches = (L.sdrgpu_launch_count() - launches0) * args.steps // (args.steps + args.warmup)
    if args.dump_outputs and not as_secondary and rank == 0:
        counts = cnt.cpu().numpy()
        dump_outputs(args.dump_outputs, {"dibits": valid_prefix(sym.cpu().numpy(), counts), "dibit_counts": counts} if hd
                     else {"audio": valid_prefix(dem.cpu().numpy(), counts), "audio_counts": counts})
    e2e = None
    if not args.device_only:
        ms_h, wall_h = timed(step_host, stream, max(3, args.steps // 2), 3)
        per = max(ms_h, wall_h) / max(3, args.steps // 2)
        e2e = {"value": channels * n * world / (per * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": per,
               "h2d_bytes_per_step": x_host.numel() * 4,
               "d2h_bytes_per_step": (sym_host.numel() if hd else dem_host.numel() * 4) + 4 * channels,
               "input": "float32 channel-domain I/Q in pinned host buffers"}
    bank.enableTiming(True)
    step()
    k_filter, k_demod = bank.lastKernelMs()
    extra_k = {}
    if hd:
        # the same step with the complete Phase 2 framing (P25P2SuperFrameDetector) running in the demodulator kernel; the
        # synthetic channels carry no sync patterns, so every symbol goes through the sync detector: the expensive state
        bank.setSyncDetector(native.SYNC_P25_PHASE2_FRAMED)
        step()
        extra_k["psk_with_phase2_framing_searching"] = bank.lastKernelMs()[1]
        bank.setSyncDetector(native.SYNC_NONE)
    bank.enableTiming(False)
    bank.dispose()
    if rank != 0:
        return None
    ms_step = ms / args.steps
    total = channels * n * world
    peak, peak_src = load_peaks()
    if hd:
        flop = channels * n * (4.0 * 154 + 40.0)
        ach = flop / (ms_step * 1e-3) / 1e12
        roof = {"bound": "fp32", "achieved": ach, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": ach / FP32_PEAK_TFLOPS,
                "traffic": load_traffic(name), "kernel": "chain: fir_agc_split_kernel + psk_multi_kernel<gardner> (whole step)",
                "kernel_ms": ms_step, "algorithmic_flop_per_step": flop,
                "peak_source": "148 SM x 128 FFMA lanes x 2 x 1.965 GHz (SURVEY.md 8d)",
                "kernels": [{"kernel": "fir_agc_split_kernel", "bound": "fp32", "ms": k_filter,
                             "achieved": channels * n * 616.0 / (k_filter * 1e-3) / 1e12, "peak": FP32_PEAK_TFLOPS,
                             "unit": "TFLOP/s", "frac": channels * n * 616.0 / (k_filter * 1e-3) / 1e12 / FP32_PEAK_TFLOPS},
                            {"kernel": "psk_multi_kernel<gardner>", "bound": "latency (serial per-symbol feedback loop)",
                             "ms": k_demod, "channels_in_launch": channels}]}
    else:
        alg = channels * n * (8.0 + 2.0)       # 8 B in + 4 B out per decimated-by-2 sample
        ach = alg / (ms_step * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": load_traffic(name), "kernel": "nbfm chain (whole step)", "kernel_ms": ms_step,
                "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                "kernels_ms": {"filters": k_filter, "demodulator": k_demod}}
    line = {"metric": METRIC, "value": total / (ms_step * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(name, 1),
            "realtime_channels": channels * world * (n / 50000.0) / (ms_step * 1e-3),
            "e2e": e2e, "gpu_launches": launches, "decode_sanity": sanity,
            "kernels_ms": dict({"filters": k_filter, "demodulator": k_demod}, **extra_k), "roofline": roof}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(name, os.cpu_count() or 1, target_seconds=6.0 if as_secondary else 10.0)
    if as_secondary:
        for key in ("metric", "n_gpus", "steps", "warmup", "higher_is_better", "scaling", "vs_baseline", "dtype", "data"):
            line.pop(key)
    return line


def run_level2(args, rank, world, local_rank, torch, dist, timed, peak, peak_src):
    """SURVEY.md 8e level 2: ONE set of tuner streams on several GPUs.  Every rank receives the same tuner buffers, runs
    the (cheap) filter bank + inverse DFT, and keeps only its contiguous slice of the polyphase bins, which it filters and
    demodulates.  No collective on the data path; strong scaling (the job is fixed, value = its input rate)."""
    import zlib
    from sdrtrunk_b200 import sharding
    dev = torch.device("cuda", local_rank)
    cfg = WORKLOADS[args.workload]
    inputs = TunerInputs(torch, dev, args.workload, 0, args.tuners)       # rank-independent seeds: the same streams everywhere
    lo, hi = sharding.bin_slice(inputs.m, rank, world)
    w = TunerWorkload(args.workload, inputs, args.tuners, local_rank, bins=(lo, hi))
    sanity = w.sanity()
    cnt = w.cnt_host.numpy().copy()
    digest = {(t, lo + c): zlib.crc32(w.sym_host.numpy()[t * (hi - lo) + c, :cnt[t * (hi - lo) + c]].tobytes())
              for t in range(args.tuners) for c in range(hi - lo)}
    w.set_format("f32")
    ms, _ = timed(w.step_device, w.stream, args.steps, args.warmup)
    gathered = [digest]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, digest)
    w.dispose()
    check = None
    if rank == 0 and args.verify:
        # the unsharded run of the same streams on this GPU: every channel's dibits must be the ones the slices produced
        full = TunerWorkload(args.workload, inputs, args.tuners, local_rank)
        full.sanity()
        fc = full.cnt_host.numpy()
        want = {(t, c): zlib.crc32(full.sym_host.numpy()[t * full.m + c, :fc[t * full.m + c]].tobytes())
                for t in range(args.tuners) for c in range(full.m)}
        got = {}
        for g in gathered:
            got.update(g)
        check = {"channels": len(want), "identical_to_unsharded": got == want}
        full.dispose()
    if rank != 0:
        return
    total = args.tuners * inputs.n_complex
    line = {"metric": METRIC, "value": total / (ms / args.steps * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args.workload, args.tuners),
                           sharding="level 2: every GPU channelizes the same tuner streams and demodulates M / N of the bins, "
                                    "no collective"),
            "bins_of_rank0": [lo, hi], "verify": check, "decode_sanity": sanity}
    print(json.dumps(line))


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from sdrtrunk_b200 import native

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    native.init(local_rank)
    dev = torch.device("cuda", local_rank)
    barrier, timed = make_timed(torch, dist, dev, world)
    peak, peak_src = load_peaks()
    cfg = WORKLOADS[args.workload]

    if cfg["kind"] == "bank":
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        line = run_bank(args.workload, args, rank, world, local_rank, torch, dist)
        if rank == 0:
            line["clocks"] = sampler.stop()
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    chain = cfg["demod"] is not None
    tuners = args.tuners if chain else 1
    if args.sharding == "level2":
        run_level2(args, rank, world, local_rank, torch, dist, timed, peak, peak_src)
        if world > 1:
            dist.destroy_process_group()
        return
    extras = (not args.no_extra) and world == 1 and args.workload == "c4fm_20m"
    curve_counts = [t for t in (1, 2, 4, 8) if t != tuners] if extras else []
    inputs = TunerInputs(torch, dev, args.workload, rank, max([tuners] + curve_counts))
    sampler = ClockSampler(local_rank)
    w = TunerWorkload(args.workload, inputs, tuners, local_rank)
    if rank == 0:
        sampler.start()
    r = measure_tuner(w, args, world, timed, full=True, capture=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.stop() if rank == 0 else None
    if "outputs" in r:
        dump_outputs(args.dump_outputs, r.pop("outputs"))
    main = summarize_tuner(w, r, peak, peak_src, args.steps, world)
    m, fs = w.m, cfg["fs"]
    w.dispose()
    del w

    secondary = {}
    if extras:
        short = argparse.Namespace(**vars(args))
        short.steps, short.warmup = max(5, args.steps // 2), 3
        curve = {str(tuners): {"value": main["value"], "ms_per_step": main["ms_per_step"], "e2e": main.get("e2e", {}).get("value"),
                               "realtime_channels": main["realtime_channels"], "kernels_ms": main["kernels_ms"]}}
        for t in curve_counts:
            wt = TunerWorkload(args.workload, inputs, t, local_rank)
            rt = measure_tuner(wt, short, world, timed, full=False)
            curve[str(t)] = {"value": rt["value"], "ms_per_step": rt["ms_per_step"],
                             "e2e": rt.get("e2e", {}).get("value"),
                             "realtime_channels": realtime_channels(rt["value"], world, m, fs), "kernels_ms": rt["kernels"]}
            wt.dispose()
            del wt
        secondary["tuners_per_gpu_curve"] = {"unit": UNIT, "note": "aggregate input MS/s of one GPU vs tuner streams batched "
                                             "into one bank (device-resident value, e2e with 8-bit host input)",
                                             "points": {k: curve[k] for k in sorted(curve, key=int)}}
        del inputs
        torch.cuda.empty_cache()
        for key, name, t in (("configs2_c4fm", "c4fm", 1), ("configs1_channelizer", "channelizer", 1)):
            inp = TunerInputs(torch, dev, name, rank, t)
            w2 = TunerWorkload(name, inp, t, local_rank)
            r2 = measure_tuner(w2, args, world, timed, full=True)
            secondary[key] = summarize_tuner(w2, r2, peak, peak_src, args.steps, world)
            w2.dispose()
            del w2, inp
            torch.cuda.empty_cache()
        short = argparse.Namespace(**vars(args))
        short.steps, short.warmup = max(5, args.steps // 2), 3
        for key, name in (("configs3_hdqpsk", "hdqpsk_4096"), ("configs0_nbfm", "nbfm_4096")):
            b = argparse.Namespace(**vars(short))
            b.no_cpu_baseline = True
            secondary[key] = run_bank(name, b, rank, world, local_rank, torch, dist, as_secondary=True)
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cores = os.cpu_count() or 1
    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, tuners),
        "realtime_channels": main["realtime_channels"] ,
        "e2e": main.get("e2e"),
        "gpu_launches": main["gpu_launches"],
        "roofline": main["roofline"],
        "kernels_ms": main["kernels_ms"],
        "cpu_baseline": cpu_baseline(args.workload, cores) if not args.no_cpu_baseline else None,
        "clocks": clocks,
    }
    for key in ("e2e_f32_input", "e2e_u8_input", "decode_sanity", "with_sync_detector", "with_frequency_corrected_channels",
                "airspy_input"):
        if key in main:
            line[key] = main[key]
    if not args.no_cpu_baseline:
        for key, name in (("configs2_c4fm", "c4fm"), ("configs1_channelizer", "channelizer"), ("configs3_hdqpsk", "hdqpsk_4096"),
                          ("configs0_nbfm", "nbfm_4096")):
            if secondary.get(key) is not None:
                secondary[key]["cpu_baseline"] = cpu_baseline(name, cores, target_seconds=5.0)
    line.update(secondary)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4fm_20m", choices=sorted(WORKLOADS))
    ap.add_argument("--tuners", type=int, default=int(os.environ.get("SDRGPU_BENCH_TUNERS", DEFAULT_TUNERS)),
                    help="tuner streams per GPU batched into one bank (chain workloads)")
    ap.add_argument("--sharding", default="level1", choices=["level1", "level2"],
                    help="level1: independent tuner streams per GPU (weak scaling); level2: the same streams on every GPU, each "
                         "keeping a slice of the polyphase bins (strong scaling)")
    ap.add_argument("--verify", action="store_true", help="level2: compare every channel's dibits with the unsharded run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements (tuner-count curve, other configs)")
    ap.add_argument("--device-only", action="store_true",
                    help="profiling aid: skip the host-buffer (e2e) passes so that every launch is a full-size one")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline workload computed as DIR/<name>.npy (float32, at "
                         "most 64 MB: a fixed, seeded sample of rows when the output is larger); the inputs are seeded, so "
                         "two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.sharding == "level2"):
        ap.error("--dump-outputs writes the outputs of the GPU arm's level1 run")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if WORKLOADS[args.workload]["kind"] != "tuner" or WORKLOADS[args.workload]["demod"] is None:
        args.tuners = 1
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
