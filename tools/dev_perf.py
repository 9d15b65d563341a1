#!/usr/bin/env python
"""Kernel-time probe used during development: cfg2 shapes (256 x 8 s), CUDA events, per cmvn mode."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import speech_lid_b200 as lid

dev = torch.device("cuda:0")
B, N = 256, 128000
modes = sys.argv[1].split(",") if len(sys.argv) > 1 else ["none", "utt", "global_accum"]
fe = lid.FrontEnd(n_mels=80)
plan = fe.make_plan([N] * B, padded=True)
g = torch.Generator(device=dev).manual_seed(1)
ins = [torch.randn(B * N, device=dev, generator=g) for _ in range(3)]
outs = [torch.empty(B, plan.t_max, 80, device=dev) for _ in range(3)]
torch.manual_seed(1234)
masks = lid.draw_masks(plan.frames, 80, 0.05, 27, 2).to(dev)
stats = torch.zeros(161, dtype=torch.float64, device=dev)
spans = fe.lib.lidfe_plan_num_spans(plan.handle)
for mode in modes:
    kw = dict(cmvn=mode)
    if mode == "global_accum":
        kw["stats_out"] = stats
    if mode in ("utt", "none"):
        kw["masks"] = masks
    for i in range(5):
        fe.featurize_packed(ins[i % 3], plan, out=outs[i % 3], **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    n = 30
    for i in range(n):
        fe.featurize_packed(ins[i % 3], plan, out=outs[i % 3], **kw)
    e1.record()
    torch.cuda.synchronize()
    print("spans=%d mode=%-13s %.1f us/step" % (spans, mode, e0.elapsed_time(e1) / n * 1e3), flush=True)
