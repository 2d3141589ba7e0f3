#!/usr/bin/env python3
"""Cost of sdrgpu_chan_set_frequency_offsets in a running stream: 8 tuners x 20 MS/s (M = 800 channels each, every
channel frequency-corrected, so pfb2_kernel mixes the oscillators in), one C4FM bank over all 6400 channels, a stream of
asynchronous submit / wait calls with two calls in flight.  A step is the host time between two consecutive wait()
returns.  Printed, with the card's name and power limit:
  steady     median step without changes;
  change     the step right after every channel of every tuner got a new nonzero offset while two calls were in flight
             (osc_reproduce_kernel rewrites two calls of look-ahead per channel on the side stream), and how long the
             set call itself took on the host;
  transition the one-time cost of switching all 800 channels of one tuner from offset 0 to nonzero (the mix tables are
             rebuilt after the work in flight): the host time of the set call and the step after it.
usage (GPU box): python tools/offset_update_time.py [seconds per call] [steady | all]   (defaults: 0.25, all)"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (the C4FM FIR taps)
from sdrtrunk_b200 import native  # noqa: E402
from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline  # noqa: E402

TUNERS, FS, M = 8, 20_000_000, 800


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 0.25
    mode = sys.argv[2] if len(sys.argv) > 2 else "all"
    native.init(0)
    n_complex = int(FS * seconds) // (1024 * (M // 2)) * (1024 * (M // 2))   # whole assembler buffers
    n_blocks = n_complex // (M // 2)
    # one pinned noise buffer per tuner, reused by every call: the step time does not depend on the samples
    g = torch.Generator().manual_seed(1)
    pinned = [(0.05 * torch.randn(2 * n_complex, generator=g)).pin_memory() for _ in range(TUNERS)]
    bufs = [t.numpy() for t in pinned]
    rates = {k: (37 if k % 2 else -53) for k in range(M)}
    chans = []
    for _ in range(TUNERS):
        ch = ComplexPolyphaseChannelizerM2(FS, 9, maxInputFloats=2 * n_complex)
        ch.setOutputChannels([([k], rates[k]) for k in range(M)])
        chans.append(ch)
    bank = Bank.preset(native.PRESET_P25_C4FM, TUNERS * M, 2.0 * FS / M, bench.fir_taps("c4fm"), max_samples_per_call=n_blocks)
    pipe = Pipeline(chans, bank)
    pipe.setChunks(8)
    pipe.setDeviceChunks(6)
    calls = [0]

    def submit():
        pipe.submit(bufs)
        calls[0] += 1

    def steps(n, before=None):
        """n steps of the stream (submit, wait) with two calls in flight; before(i) runs before submit i"""
        out, last = [], None
        for i in range(n):
            if before:
                before(i)
            submit()
            pipe.wait()
            now = time.perf_counter()
            if last is not None:
                out.append(1e3 * (now - last))
            last = now
        return out

    submit()   # one call in flight from here on
    steps(4)
    print("card: %s (name, power limit, max SM clock)" % card())
    print("workload: %d tuners x %.0f MS/s, M = %d, every channel corrected, C4FM bank of %d channels, %d blocks "
          "(%.2f s) per call, submit / wait with two calls in flight" % (TUNERS, FS / 1e6, M, TUNERS * M, n_blocks, seconds))
    steady = steps(21)
    print("steady     median step %.3f ms (min %.3f, max %.3f, %d steps)" % (np.median(steady), min(steady), max(steady),
                                                                             len(steady)))
    if mode == "steady":
        pipe.wait()
        return
    after, host = [], []
    for r in range(6):
        t_set = []

        def change(i, r=r):
            if i == 1:   # calls 0 and the one before it are in flight
                t0 = time.perf_counter()
                for k, ch in enumerate(chans):
                    ch.setFrequencyOffsets({c: (41 + r + c % 7 + k) * (1 if c % 2 else -1) for c in range(M)})
                t_set.append(1e3 * (time.perf_counter() - t0))
        s = steps(4, change)
        after.append(max(s))   # the steps around the first call with the new offsets
        host.append(t_set[0])
        print("change %d   steps %s ms; set calls (8 tuners x 800 channels) %.3f ms on the host" %
              (r, " ".join("%.3f" % v for v in s), t_set[0]))
    print("change     median of the longest step around a change of every channel %.3f ms (steady %.3f); host time of the 8 set calls "
          "%.3f ms" % (np.median(after), np.median(steady), np.median(host)))
    # one tuner: every channel to 0, then back to nonzero (the rebuild path both ways)
    for r in range(3):
        t0 = time.perf_counter()
        chans[0].setFrequencyOffsets({c: 0 for c in range(M)})
        t_off = 1e3 * (time.perf_counter() - t0)
        s_off = steps(3)
        t0 = time.perf_counter()
        chans[0].setFrequencyOffsets({c: 29 + c % 5 for c in range(M)})
        t_on = 1e3 * (time.perf_counter() - t0)
        s_on = steps(3)
        print("transition %d: all 800 channels of tuner 0 -> 0: set %.3f ms, steps %s; 0 -> nonzero: set %.3f ms, steps %s" %
              (r, t_off, " ".join("%.3f" % v for v in s_off), t_on, " ".join("%.3f" % v for v in s_on)))
    pipe.wait()
    pipe.dispose()


if __name__ == "__main__":
    main()
