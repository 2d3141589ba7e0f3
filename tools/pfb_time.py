#!/usr/bin/env python3
"""Channelizer kernel time alone, with CUDA events, at the bench's sizes: one second of a 10 MS/s tuner (M = 400) and of
a 20 MS/s tuner (M = 800), float and signed 8-bit input, device-resident input and output rows.  For each case it prints
the time per call and a CRC-32 of the output rows of the first call on a fresh handle, so that two builds run one after
the other compare both time and bits.  usage (GPU box): python tools/pfb_time.py [calls]"""
import ctypes as C
import os
import sys
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from sdrtrunk_b200 import native  # noqa: E402
from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2  # noqa: E402


def run(fs, fmt, calls):
    dev = torch.device("cuda", 0)
    n_complex = int(fs)
    g = torch.Generator(device=dev)
    g.manual_seed(12345)
    x = torch.randn(2 * n_complex, generator=g, device=dev, dtype=torch.float32) * 0.1
    if fmt == "s8":   # SignedByteSampleConverter: value / 128
        x = torch.clamp(torch.round(x * 128.0), -128, 127).to(torch.int8)
    stream = torch.cuda.Stream(device=dev)
    ch = ComplexPolyphaseChannelizerM2(fs, 9, device=0, maxInputFloats=2 * n_complex)
    ch.setStream(stream.cuda_stream)
    ch.setSampleFormat(fmt)
    L = native.lib()
    m = L.sdrgpu_channel_count_for_rate(C.c_double(fs))
    n_blocks = L.sdrgpu_chan_blocks_for(ch._h, 2 * n_complex)
    out = torch.empty((m, 2 * n_blocks), dtype=torch.float32, device=dev)

    def call():
        native.check(L.sdrgpu_chan_process(ch._h, C.c_void_p(x.data_ptr()), 2 * n_complex, native.DEVICE,
                                           C.c_void_p(out.data_ptr()), 2 * n_blocks, native.DEVICE,
                                           native.LAYOUT_CHANNELS, None))

    with torch.cuda.stream(stream):
        call()
        stream.synchronize()
        crc = zlib.crc32(out.cpu().numpy().tobytes())
        for _ in range(3):
            call()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        for _ in range(calls):
            call()
        stop.record(stream)
        stop.synchronize()
    ms = start.elapsed_time(stop) / calls
    ch.dispose()
    print("M = %d  %-3s  %d samples  %.4f ms per call  crc %08x" % (m, fmt, n_complex, ms, crc), flush=True)


def main():
    calls = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    native.init(0)
    for fs in (10e6, 20e6):
        for fmt in ("f32", "s8"):
            run(fs, fmt, calls)


if __name__ == "__main__":
    main()
