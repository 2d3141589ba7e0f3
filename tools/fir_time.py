#!/usr/bin/env python3
"""FIR + block AGC time of a C4FM bank (72 taps, 1024-sample AGC buffers) by channel count, for both FIR kernels.
fir_agc_split_kernel runs the bank as it is.  For fir_agc_kernel the launch is held to 6 CTAs per SM
(sdrgpu_set_tuning THROTTLE_ALWAYS + FIR_CTAS_PER_SM): that is the kernel's own register-bound occupancy (80 registers
x 128 threads), so the shape is unchanged, while the larger shared-memory request takes the launch off the split kernel.
usage (GPU box): python tools/fir_time.py [channels ...]"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from sdrtrunk_b200 import native  # noqa: E402
from sdrtrunk_b200.dsp import Bank  # noqa: E402
from psk_layout_sweep import oracle_taps  # noqa: E402

KERNELS = (("fir_agc_split_kernel", 0), ("fir_agc_kernel", 6))   # (kernel, FIR CTAs per SM: 0 = not throttled)


def main():
    native.init(0)
    lib = native.lib()
    rng = np.random.default_rng(0)
    n = 12 * 1024
    fir = oracle_taps()
    try:
        for c in [int(a) for a in sys.argv[1:]] or [800, 6400]:
            x = rng.standard_normal((c, 2 * n), dtype=np.float32) * 0.1
            bank = Bank.preset(native.PRESET_P25_C4FM, c, 50000.0, fir, max_samples_per_call=n)
            bank.enableTiming(True)
            for kernel, ctas in KERNELS:
                native.check(lib.sdrgpu_set_tuning(native.TUNE_THROTTLE_ALWAYS, 1 if ctas else 0))
                native.check(lib.sdrgpu_set_tuning(native.TUNE_FIR_CTAS_PER_SM, ctas))
                best = 1e9
                for _ in range(4):
                    bank.process(x)
                    best = min(best, bank.lastKernelMs()[0])
                print("%5d channels x %d samples: %-20s %.4f ms" % (c, n, kernel, best), flush=True)
            bank.dispose()
    finally:
        native.check(lib.sdrgpu_set_tuning(native.TUNE_THROTTLE_ALWAYS, 0))
        native.check(lib.sdrgpu_set_tuning(native.TUNE_FIR_CTAS_PER_SM, 0))


if __name__ == "__main__":
    main()
