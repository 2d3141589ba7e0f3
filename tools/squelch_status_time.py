#!/usr/bin/env python3
"""Cost of the squelch status bytes (sdrgpu_bank_set_squelch_reporting) on bench.py's nbfm_4096 workload: 4096 NBFM
channel-domain streams at 50 kHz, 24 Ki samples per channel per call (decimate by 2 -> 45-tap FIR -> squelching FM
discriminator, nbfm_fused_kernel), device-resident input and outputs.  Two banks of the same configuration, one with
reporting off and one with it on, are called alternately in one process; each call's device time comes from CUDA events
around it on the banks' stream.  Prints the card's name and power limit, the per-call device time of each variant, and
whether the two produced bit-identical audio on every call.
usage (GPU box): python tools/squelch_status_time.py [reps]"""
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (the nbfm_4096 workload's signal and FIR taps)
from sdrtrunk_b200 import native  # noqa: E402
from sdrtrunk_b200.dsp import Bank  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 40
    cfg = bench.WORKLOADS["nbfm_4096"]
    channels, n = cfg["channels"], cfg["samples"]
    native.init(0)
    L = native.lib()
    dev = torch.device("cuda", 0)
    x = bench.synth_nbfm_channels(torch, dev, channels, n, seed=5)
    fir = bench.fir_taps("nbfm")
    stream = torch.cuda.Stream(device=dev)
    blocks = n // 1024
    variants = {}
    for name, report in (("off", False), ("on", True)):
        bank = Bank.preset(native.PRESET_NBFM, channels, 50000.0, fir, max_samples_per_call=n)
        bank.setStream(stream.cuda_stream)
        if report:
            native.check(L.sdrgpu_bank_set_squelch_reporting(bank._h, 1))
        variants[name] = dict(bank=bank, times=[],
                              dem=torch.zeros((channels, n // 2), dtype=torch.float32, device=dev),
                              sym=torch.zeros((channels, blocks), dtype=torch.uint8, device=dev) if report else None,
                              cnt=torch.zeros(channels, dtype=torch.int32, device=dev))
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None   # noqa: E731
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def call(v):
        with torch.cuda.stream(stream):
            start.record(stream)
            native.check(L.sdrgpu_bank_process(v["bank"]._h, vp(x), 2 * n, n, native.DEVICE, vp(v["sym"]), blocks,
                                               vp(v["dem"]), n // 2, vp(v["cnt"]), native.DEVICE))
            stop.record(stream)
        stop.synchronize()
        return start.elapsed_time(stop)

    identical = True
    for i in range(reps + 3):
        order = ("off", "on") if i % 2 == 0 else ("on", "off")
        for name in order:
            ms = call(variants[name])
            if i >= 3:
                variants[name]["times"].append(ms)
        identical &= torch.equal(variants["off"]["dem"].view(torch.int32), variants["on"]["dem"].view(torch.int32))
    st = variants["on"]["sym"].cpu().numpy()
    print("card: %s (name, power limit, max SM clock)" % card())
    print("workload: nbfm_4096, %d channels x %d samples at 50 kHz per call (%d assembler buffers), device input and "
          "outputs; %d timed calls per variant, alternated" % (channels, n, blocks, reps))
    for name in ("off", "on"):
        t = np.array(variants[name]["times"])
        print("reporting %-3s  device time per call: median %.4f ms  (min %.4f, max %.4f)" %
              (name, np.median(t), t.min(), t.max()))
    off, on = np.median(variants["off"]["times"]), np.median(variants["on"]["times"])
    print("on / off = %.4f (%+.2f %%); audio bit-identical on every call: %s" % (on / off, 100.0 * (on / off - 1.0), identical))
    print("statuses of the last call: %d channels muted (MUTE), %d open (UNMUTE), %d with a change in the last buffer" %
          (int(np.sum(st[:, -1] & 3 == native.SQUELCH_MUTE)), int(np.sum(st[:, -1] & 3 == native.SQUELCH_UNMUTE)),
           int(np.sum(st[:, -1] & native.SQUELCH_CHANGED != 0))))
    for v in variants.values():
        v["bank"].dispose()


if __name__ == "__main__":
    main()
