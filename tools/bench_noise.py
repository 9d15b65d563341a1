#!/usr/bin/env python
"""Cost of on-device additive noise (FrontEnd.add_noise / lidfe_add_noise) on one GPU: CUDA events, rotating input
buffers larger than L2 in total.  One JSON line per measurement, the card's name and power limit first.

  * the add_noise kernel alone on the cfg2 shape (256 x 8 s = 32.77 M samples): bank source (64 clips of 10 s) and
    Gaussian source, each with and without normalize, and int16 input.  Each line carries the bytes the pass needs
    (x read once, the noise read once, y written once; the later passes re-read x and the noise from L2) and the time
    that traffic takes at the data sheet's 7.7 TB/s;
  * the cfg2 chain (fbank + SpecAugment + per-utterance CMVN) with and without add_noise in front;
  * a ragged DeviceCollate training step (host waveforms in, masks, CMVN) with noise augmentation on and off.

usage: python tools/bench_noise.py [steps]"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import speech_lid_b200 as lid

HBM_TBPS = 7.7          # data sheet, HGX B200, one GPU
STEPS = int(sys.argv[1]) if len(sys.argv) > 1 else 100
B, N = 256, 128000


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
    except Exception as e:          # the timing lines still carry the torch device name
        name, power, clock = torch.cuda.get_device_name(0), "unknown (%s)" % type(e).__name__, "unknown"
    return {"card": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name(0)}


def timed(fn, nbuf, steps=None, warmup=10):
    steps = steps or STEPS
    for i in range(warmup):
        fn(i % nbuf)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i % nbuf)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    torch.cuda.set_device(0)
    info = card()
    print(json.dumps(info), flush=True)
    dev = torch.device("cuda:0")
    fe = lid.FrontEnd(n_mels=80)
    plan = fe.make_plan([N] * B, padded=True)
    g = torch.Generator(device=dev).manual_seed(1)
    nbuf = 3                                                    # 3 x 131 MB of input: more than L2 holds
    ins = [torch.randn(B * N, device=dev, generator=g) for _ in range(nbuf)]
    ins16 = [(w * 3000).clamp(-32768, 32767).to(torch.int16) for w in ins]
    outs = [torch.zeros(B * N, device=dev) for _ in range(nbuf)]
    hg = torch.Generator().manual_seed(3)
    bank = lid.NoiseBank([torch.randn(160000, generator=hg) for _ in range(64)], device=dev)
    draw = lid.draw_noise(B, (0.0, 20.0), 1.0, bank, hg)
    tab, snr = lid.noise.noise_table(draw, bank, B)
    tab, snr = tab.to(dev), snr.to(dev)
    lib = lid.load_library()

    def kernel(src, use_bank, normalize):
        def launch(i):
            x = src[i]
            rc = lib.lidfe_add_noise(fe.handle, plan.handle, x.data_ptr(), int(x.dtype == torch.int16), 1.0 / 32768,
                                     outs[i].data_ptr(), bank.data.data_ptr() if use_bank else None,
                                     bank.data.numel(), tab.data_ptr(), snr.data_ptr(), draw.seed, int(normalize),
                                     torch.cuda.current_stream().cuda_stream)
            assert rc == 0, rc
        return launch

    samples = B * N
    for label, src, use_bank, normalize, bps in (
            ("bank, float32", ins, True, False, 12), ("bank, float32, normalize", ins, True, True, 12),
            ("gaussian, float32", ins, False, False, 8), ("gaussian, float32, normalize", ins, False, True, 8),
            ("bank, int16", ins16, True, False, 10), ("bank, int16, normalize", ins16, True, True, 10),
            ("gaussian, int16", ins16, False, False, 6)):
        ms = timed(kernel(src, use_bank, normalize), nbuf)
        floor_us = samples * bps / (HBM_TBPS * 1e12) * 1e6
        print(json.dumps({"pass": "add_noise kernel: " + label, "utterances": B, "samples": N, "us": round(ms * 1e3, 1),
                          "bytes_per_sample": bps, "mbytes": round(samples * bps / 1e6, 1),
                          "hbm_floor_us": round(floor_us, 1), "x_floor": round(ms * 1e3 / floor_us, 2),
                          "card": info["card"], "power_limit": info["power_limit"]}), flush=True)

    # the cfg2 step with and without the noise in front (the public API: table upload included)
    torch.manual_seed(0)
    masks = lid.draw_masks(plan.frames, 80, 0.05, 27, 2).cuda()
    feats = [torch.empty(B, plan.t_max, 80, device=dev) for _ in range(nbuf)]

    def plain(i):
        fe.featurize_packed(ins[i], plan, out=feats[i], masks=masks, cmvn="utt")

    def noisy(i):
        y = fe.add_noise(ins[i], plan, draw, bank=bank, out=outs[i])
        fe.featurize_packed(y, plan, out=feats[i], masks=masks, cmvn="utt")

    t_plain, t_noisy = [], []
    for _ in range(3):                                          # alternate: other work shares the host
        t_plain.append(timed(plain, nbuf))
        t_noisy.append(timed(noisy, nbuf))
    print(json.dumps({"pass": "cfg2 chain (fbank + SpecAugment + per-utterance CMVN), 256 x 8 s",
                      "plain_ms": [round(t, 4) for t in t_plain], "with_add_noise_ms": [round(t, 4) for t in t_noisy],
                      "card": info["card"], "power_limit": info["power_limit"]}), flush=True)

    # a ragged training step through DeviceCollate: host waveforms of 2-12 s, 2 masks, per-utterance CMVN
    rg = torch.Generator().manual_seed(5)
    lens = [int(v) for v in torch.randint(32000, 192000, (128,), generator=rg)]
    batch = [(torch.randn(1, n, generator=rg) * 0.1, torch.tensor([1, 2]), "u%d" % i, "en") for i, n in enumerate(lens)]
    l2i = {"en": 0}
    aug = lid.NoiseAugment(bank, (0.0, 20.0), p=1.0, generator=torch.Generator().manual_seed(6))
    dc_plain = lid.DeviceCollate(fe, l2i, train=True, mask_times=2, cmvn="utt")
    dc_noisy = lid.DeviceCollate(fe, l2i, train=True, mask_times=2, cmvn="utt", noise=aug)

    def step_ms(dc, steps=20):
        for _ in range(3):
            dc(batch)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            dc(batch)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / steps

    r_plain, r_noisy = [], []
    for _ in range(3):
        r_plain.append(step_ms(dc_plain))
        r_noisy.append(step_ms(dc_noisy))
    print(json.dumps({"pass": "DeviceCollate ragged step, 128 utterances of 2-12 s (%.0f s of audio), host in" % (sum(lens) / 16000),
                      "noise_off_ms": [round(t, 3) for t in r_plain], "noise_on_ms": [round(t, 3) for t in r_noisy],
                      "card": info["card"], "power_limit": info["power_limit"]}), flush=True)


if __name__ == "__main__":
    main()
