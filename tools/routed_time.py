#!/usr/bin/env python3
"""A mixed deployment on one GPU: 8 tuners x 20 MS/s (M = 800, signed 8-bit samples, 1 s per tuner per call), every
tuner's 800 channels split between a C4FM bank (640 per tuner, 5120 rows) and an NBFM bank (160 per tuner, 1280 rows),
run as
  (a) one routed pipeline (sdrgpu_pipeline_create_routed: one channelizer pass per tuner feeds both banks), and
  (b) two one-bank pipelines (sdrgpu_pipeline_create_multi) whose channelizers select the same split -- every tuner
      buffer is channelized twice and, with host input, copied to the device twice.
Device-resident and pinned host input; calls of (a) and (b) alternate.  Prints the card, its power limit and maximum SM
clock, the time per call of each, and whether (a) and (b) produced identical dibits, counts and audio on every call.
usage (GPU box): python tools/routed_time.py [reps]"""
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle  # noqa: E402  (the reference's filter designs: the C4FM and NBFM FIR taps)
from sdrtrunk_b200 import native  # noqa: E402
from sdrtrunk_b200.dsp import Bank, ComplexPolyphaseChannelizerM2, Pipeline  # noqa: E402

TUNERS, FS, M = 8, 20e6, 800
NBFM_BIN = [b % 5 == 4 for b in range(M)]          # 160 of 800 bins per tuner


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def channelizers(bins, n_complex):
    out = []
    for _ in range(TUNERS):
        ch = ComplexPolyphaseChannelizerM2(FS, 9, maxInputFloats=2 * n_complex)
        ch.setSampleFormat("s8")
        ch.setChannels(bins)
        out.append(ch)
    return out


def banks(n_channel_samples):
    c4 = Bank.preset(native.PRESET_P25_C4FM, TUNERS * 640, 50000.0, oracle.c4fm_baseband_taps(),
                     max_samples_per_call=n_channel_samples)
    fm = Bank.preset(native.PRESET_NBFM, TUNERS * 160, 50000.0, oracle.nbfm_iq_taps(), max_samples_per_call=n_channel_samples)
    return c4, fm


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    native.init(0)
    L = native.lib()
    dev = torch.device("cuda", 0)
    n_complex = int(FS)
    g = torch.Generator(device=dev)
    g.manual_seed(2024)
    x_dev = [torch.clamp(torch.round(torch.randn(2 * n_complex, generator=g, device=dev) * 20.0), -128, 127).to(torch.int8)
             for _ in range(TUNERS)]
    x_host = [x.cpu().pin_memory() for x in x_dev]
    all_bins = list(range(M))
    c4_bins = [b for b in all_bins if not NBFM_BIN[b]]
    fm_bins = [b for b in all_bins if NBFM_BIN[b]]
    n_ch = n_complex // (M // 2)

    a_chans = channelizers(all_bins, n_complex)
    a_banks = banks(n_ch)
    route = [1 if NBFM_BIN[b] else 0 for _ in range(TUNERS) for b in all_bins]
    a = Pipeline(a_chans, banks=list(a_banks), route=route)
    b_banks = banks(n_ch)
    b_c4 = Pipeline(channelizers(c4_bins, n_complex), b_banks[0])
    b_fm = Pipeline(channelizers(fm_bins, n_complex), b_banks[1])

    # outputs: pinned host buffers, one set per variant
    blocks = n_ch // 1024 + 1
    stride = blocks * 1024 // 3 + 16
    fm_len = blocks * 512

    def outputs():
        return dict(sym=torch.zeros((TUNERS * 640, stride), dtype=torch.uint8).pin_memory(),
                    cnt=torch.zeros(TUNERS * 640, dtype=torch.int32).pin_memory(),
                    dem=torch.zeros((TUNERS * 160, fm_len), dtype=torch.float32).pin_memory(),
                    fcnt=torch.zeros(TUNERS * 160, dtype=torch.int32).pin_memory())

    oa, ob = outputs(), outputs()
    routed_out = (native.BankOutput * 2)()
    routed_out[0].symbols, routed_out[0].symbol_stride, routed_out[0].counts = oa["sym"].data_ptr(), stride, oa["cnt"].data_ptr()
    routed_out[1].demod, routed_out[1].demod_stride_floats, routed_out[1].counts = oa["dem"].data_ptr(), fm_len, oa["fcnt"].data_ptr()

    def ptrs(xs):
        return (C.c_void_p * TUNERS)(*[t.data_ptr() for t in xs])

    def run_a(xs, mem):
        native.check(L.sdrgpu_pipeline_process_routed(a._h, ptrs(xs), 2 * n_complex, mem, routed_out, native.HOST))

    def run_b(xs, mem):
        p = ptrs(xs)
        native.check(L.sdrgpu_pipeline_process_multi(b_c4._h, p, 2 * n_complex, mem, C.c_void_p(ob["sym"].data_ptr()), stride,
                                                     None, 0, C.c_void_p(ob["cnt"].data_ptr()), native.HOST))
        native.check(L.sdrgpu_pipeline_process_multi(b_fm._h, p, 2 * n_complex, mem, None, 0, C.c_void_p(ob["dem"].data_ptr()),
                                                     fm_len, C.c_void_p(ob["fcnt"].data_ptr()), native.HOST))

    def same():
        ok = torch.equal(oa["cnt"], ob["cnt"]) and torch.equal(oa["fcnt"], ob["fcnt"]) and torch.equal(oa["dem"], ob["dem"])
        cnt = oa["cnt"].numpy()
        sa, sb = oa["sym"].numpy(), ob["sym"].numpy()
        return ok and all(np.array_equal(sa[r, :cnt[r]], sb[r, :cnt[r]]) for r in range(cnt.size))

    print("card: %s (name, power limit, max SM clock)" % card())
    print("workload: %d tuners x %.0f MS/s, M = %d, s8 input, %d complex samples per tuner per call; C4FM bank %d rows, "
          "NBFM bank %d rows; %d timed calls per variant and input" % (TUNERS, FS / 1e6, M, n_complex, TUNERS * 640,
                                                                     TUNERS * 160, reps))
    for name, xs, mem in (("device input", x_dev, native.DEVICE), ("host input (pinned)", x_host, native.HOST)):
        times = {"a": [], "b": []}
        identical = True
        for i in range(reps + 2):
            for key, fn in (("a", run_a), ("b", run_b)) if i % 2 == 0 else (("b", run_b), ("a", run_a)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(xs, mem)
                torch.cuda.synchronize()
                if i >= 2:
                    times[key].append((time.perf_counter() - t0) * 1e3)
            identical &= same()
        ma, mb = np.median(times["a"]), np.median(times["b"])
        print("%-20s (a) routed pipeline      median %7.2f ms per call  (min %7.2f, max %7.2f)" %
              (name, ma, min(times["a"]), max(times["a"])))
        print("%-20s (b) two pipelines        median %7.2f ms per call  (min %7.2f, max %7.2f)" %
              (name, mb, min(times["b"]), max(times["b"])))
        print("%-20s (a) / (b) = %.3f; outputs of (a) and (b) identical on every call: %s" % (name, ma / mb, identical))
    for p in (a, b_c4, b_fm):
        p.dispose()


if __name__ == "__main__":
    main()
