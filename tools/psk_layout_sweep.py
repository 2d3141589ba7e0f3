#!/usr/bin/env python3
"""Demodulator kernel time by bank size and lanes per channel (C4FM, decision directed): the data behind the
automatic layout choice in psk.cu.  usage (GPU box): python tools/psk_layout_sweep.py"""
import os
import sys

import numpy as np
import scipy.signal as ss

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import siggen as sg  # noqa: E402
from sdrtrunk_b200 import native  # noqa: E402
from sdrtrunk_b200.dsp import Bank  # noqa: E402


def oracle_taps():
    """the C4FM decoder's own baseband filter (libsdrgpu's restatement of RemezFIRFilterDesigner)"""
    from sdrtrunk_b200.dsp import FilterFactory, FIRFilterSpecification
    return FilterFactory.getTaps(FIRFilterSpecification.lowPassBuilder().sampleRate(50000.0).passBandCutoff(5100)
                                 .passBandRipple(0.01).stopBandStart(6500).stopBandRipple(0.01).build())


def main():
    native.init(0)
    rng = np.random.default_rng(0)
    n = 24 * 1024
    fir = oracle_taps()
    base = []
    for k in range(8):
        dib = rng.integers(0, 4, int(n * 4800 / 50000) + 8)
        z = sg.c4fm(dib, carrier_offset=rng.uniform(-200, 200), timing_phase=rng.uniform(0, 1), n_samples=n)
        base.append(sg.interleave(z + sg.awgn(rng, n, 0.03)))
    base = np.stack(base)
    counts = [int(a) for a in sys.argv[1:]] or [400, 800, 1200, 1600, 2400, 3200, 4800, 6400]
    for c in counts:
        x = np.tile(base, (c // 8, 1))
        row = []
        for lanes in (32, 16, 8, 4, 2, 1):
            bank = Bank.preset(native.PRESET_P25_C4FM, c, 50000.0, fir, max_samples_per_call=n)
            bank.setDemodulatorLanes(lanes)
            bank.enableTiming(True)
            best = 1e9
            for _ in range(3):
                bank.process(x)
                best = min(best, bank.lastKernelMs()[1])
            row.append(best)
            bank.dispose()
        print("%5d channels: 32 lanes %.3f ms, 16 lanes %.3f ms, 8x2 %.3f ms, 4x3 %.3f ms, 2x6 %.3f ms, 1 lane %.3f ms" % (c, *row),
              flush=True)


if __name__ == "__main__":
    main()
