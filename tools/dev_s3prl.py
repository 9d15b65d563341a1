#!/usr/bin/env python
"""Development: throughput of speech_lid_b200.S3prlFBank (the wav2vec-exp FBank variant) on 256 x 8 s, per kernel path of
the windowed-DFT GEMM (LIDFE_RESAMPLE_TC: tcgen05 or FP32)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import speech_lid_b200 as lid

B, N = 256, 128000
g = torch.Generator(device="cuda").manual_seed(1)
wavs = [torch.randn(N, device="cuda", generator=g) for _ in range(B)]
for kind in ("tc", "fp32"):
    os.environ["LIDFE_RESAMPLE_TC"] = "1" if kind == "tc" else "0"
    fb = lid.S3prlFBank(80, 640)
    for _ in range(3):
        fb.forward_list(wavs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        fb.forward_list(wavs)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    print("S3prlFBank(80, 640) %-4s: %.3f ms per 256 x 8 s (incl. torch.cat of the inputs) = %.2f M audio-s/s" % (kind, ms, B * 8.0 / ms / 1e3), flush=True)
