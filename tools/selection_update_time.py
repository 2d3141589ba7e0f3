#!/usr/bin/env python3
"""Cost of sdrgpu_chan_update_selection in a running stream: 8 tuners x 20 MS/s (M = 800 channels each), one C4FM bank
over all 6400 channels (sdrgpu_pipeline_create_multi), a stream of asynchronous submit / wait calls with two calls in
flight.  A step is the host time between two consecutive wait() returns.  Printed, with the card's name and power limit:
  steady  median step without edits;
  update  an edit that retunes k = 1, 8 or 800 channels of every tuner to other bins (the row count stays), issued while
          two calls are in flight: the host time of the 8 update calls and the steps around it.  The edit is undone
          the same way before the next one;
  select  the same retune done with sdrgpu_chan_select (every channel of the tuner restarts), for comparison.
With --corrected every channel has a frequency offset (pfb2_kernel mixes the oscillators in until an edit moves bins
out of order); without it every channel is plain (the identity direct store).
usage (GPU box): python tools/selection_update_time.py [--corrected] [--steady-only] [seconds per call]"""
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
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    corrected = "--corrected" in sys.argv
    seconds = float(args[0]) if args else 0.25
    native.init(0)
    n_complex = int(FS * seconds) // (1024 * (M // 2)) * (1024 * (M // 2))   # whole assembler buffers
    n_blocks = n_complex // (M // 2)
    g = torch.Generator().manual_seed(1)
    pinned = [(0.05 * torch.randn(2 * n_complex, generator=g)).pin_memory() for _ in range(TUNERS)]
    bufs = [t.numpy() for t in pinned]
    offset = (lambda c: 37 + c % 7 if c % 2 else -53 - c % 5) if corrected else (lambda c: 0)
    base = [([c], offset(c)) for c in range(M)]
    chans = []
    for _ in range(TUNERS):
        ch = ComplexPolyphaseChannelizerM2(FS, 9, maxInputFloats=2 * n_complex)
        ch.setOutputChannels(base)
        chans.append(ch)
    bank = Bank.preset(native.PRESET_P25_C4FM, TUNERS * M, 2.0 * FS / M, bench.fir_taps("c4fm"), max_samples_per_call=n_blocks)
    pipe = Pipeline(chans, bank)
    pipe.setChunks(8)
    pipe.setDeviceChunks(6)

    def steps(n, before=None):
        """n steps of the stream (submit, wait) with two calls in flight; before(i) runs before submit i"""
        out, last = [], None
        for i in range(n):
            if before:
                before(i)
            pipe.submit(bufs)
            pipe.wait()
            now = time.perf_counter()
            if last is not None:
                out.append(1e3 * (now - last))
            last = now
        return out

    pipe.submit(bufs)   # one call in flight from here on
    steps(4)
    print("card: %s (name, power limit, max SM clock)" % card())
    print("workload: %d tuners x %.0f MS/s, M = %d, %s channels, C4FM bank of %d channels, %d blocks (%.2f s) per call, "
          "submit / wait with two calls in flight" % (TUNERS, FS / 1e6, M, "corrected" if corrected else "plain",
                                                     TUNERS * M, n_blocks, seconds))
    steady = steps(21)
    print("steady   median step %.3f ms (min %.3f, max %.3f, %d steps)" % (np.median(steady), min(steady), max(steady),
                                                                           len(steady)))
    if "--steady-only" in sys.argv:
        pipe.wait()
        pipe.dispose()
        return

    def retuned(k):
        """channels 0 .. k - 1 move to the next bin up (setPolyphaseChannelIndices); offsets stay"""
        return [([(c + 1) % M], offset(c)) if c < k else e for c, e in enumerate(base)]

    keep = list(range(M))
    for how in ("update", "select"):
        for k in (1, 8, 800):
            hosts, around = [], []
            for r in range(3):
                for sel in (retuned(k), base):
                    t = []

                    def edit(i, sel=sel):
                        if i == 1:   # two calls in flight
                            t0 = time.perf_counter()
                            for ch in chans:
                                if how == "update":
                                    ch.updateOutputChannels(sel, keep)
                                else:
                                    ch.setOutputChannels(sel)
                            t.append(1e3 * (time.perf_counter() - t0))
                    s = steps(4, edit)
                    hosts.append(t[0])
                    around.append(s)
            print("%s k=%-3d host time of the 8 calls: median %.3f ms (%s); steps around: %s" %
                  (how, k, np.median(hosts), " ".join("%.2f" % v for v in hosts),
                   " | ".join(" ".join("%.2f" % v for v in s) for s in around)))
    pipe.wait()
    pipe.dispose()


if __name__ == "__main__":
    main()
