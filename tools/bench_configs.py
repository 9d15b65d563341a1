#!/usr/bin/env python
"""Device-resident throughput of the other BASELINE configs / branches on one GPU (CUDA events, rotating buffers):
cfg1 (32 x 3 s fbank), cfg2 without CMVN, cfg3 (512 x 4 s MFCC-40 of 80) and MFCC-40 of 60 mel, the default
MelSpectrogram+dB branch on the cfg2 shape, int16 input, the resampler.  One JSON line each; informational (bench.py carries the headline)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import speech_lid_b200 as lid


def run(name, fe, B, N, steps=None, warmup=10, dtype=torch.float32, quiet_tail=False, **kw):
    if ONLY and ONLY not in name:
        return
    steps = steps or STEPS
    dev = fe.device
    plan = fe.make_plan([N] * B, padded=True)
    g = torch.Generator(device=dev).manual_seed(1)
    nbuf = max(3, int(400e6 // (B * N * 4)) if B * N * 4 < 130e6 else 3)
    ins = []
    for _ in range(nbuf):
        w = torch.randn(B * N, device=dev, generator=g)
        if quiet_tail:                       # last quarter of every utterance 100 dB down: AmplitudeToDB's clamp is active there
            w.view(B, N)[:, 3 * N // 4:] *= 1e-5
        ins.append((w * 3000).clamp(-32768, 32767).to(torch.int16) if dtype == torch.int16 else w)
    outs = [torch.empty(B, plan.t_max, fe.n_out, device=dev) for _ in range(nbuf)]
    for i in range(warmup):
        fe.featurize_packed(ins[i % nbuf], plan, out=outs[i % nbuf], **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fe.featurize_packed(ins[i % nbuf], plan, out=outs[i % nbuf], **kw)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    audio_s = B * N / 16000.0
    print(json.dumps({"config": name, "utterances": B, "samples": N, "frames": plan.total_frames, "ms_per_step": round(ms, 5),
                      "audio_s_per_s": round(audio_s / (ms * 1e-3), 1), "rotating_sets": nbuf}), flush=True)


ONLY = sys.argv[1] if len(sys.argv) > 1 else ""      # substring filter on the config name, e.g. "cfg3"
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 100


def main():
    torch.cuda.set_device(0)
    fb = lid.FrontEnd(n_mels=80)
    run("cfg1: 80-dim kaldi fbank, 32 x 3 s", fb, 32, 48000)
    run("cfg2 shape, kaldi fbank only (no CMVN, no masks), 256 x 8 s", fb, 256, 128000)
    masks = lid.draw_masks([798] * 256, 80, 0.05, 27, 2).cuda()      # resident, like the waveforms
    run("cfg2 shape, kaldi fbank + SpecAugment in the epilogue (no CMVN), 256 x 8 s", fb, 256, 128000, masks=masks)
    run("cfg2: kaldi fbank + SpecAugment + per-utterance CMVN, 256 x 8 s", fb, 256, 128000, masks=masks, cmvn="utt")
    mf = lid.FrontEnd(n_mels=80, n_ceps=40)
    run("cfg3: 40 MFCC of 80 mel (DCT epilogue), 512 x 4 s", mf, 512, 64000)
    run("MFCC-40 of 60 mel (n_mels % 8 == 4: half a last k-step in the DCT), 512 x 4 s", lid.FrontEnd(n_mels=60, n_ceps=40), 512, 64000)
    ms = lid.FrontEnd(kind="melspec_db", pad=16)
    run("default branch: MelSpectrogram + AmplitudeToDB(top_db=80), pad 16, 256 x 8 s (white noise: nothing to clamp)", ms, 256, 128000)
    run("default branch, last quarter of every utterance 100 dB down (clamp active in a quarter of the row blocks)", ms, 256,
        128000, quiet_tail=True)
    i16 = lid.FrontEnd(n_mels=80, in_dtype=torch.int16, in_scale=1.0 / 32768.0)
    run("kaldi fbank from int16 samples (2 B/sample read), 256 x 8 s", i16, 256, 128000, dtype=torch.int16)
    pf = lid.FrontEnd(n_mels=80, precise=True)
    run("precise mode (float64 kernel): kaldi fbank only, 256 x 8 s", pf, 256, 128000)
    run("precise mode: cfg2 (fbank + SpecAugment + per-utterance CMVN), 256 x 8 s", pf, 256, 128000, masks=masks, cmvn="utt")
    run("precise mode: cfg3 (40 MFCC of 80 mel), 512 x 4 s", lid.FrontEnd(n_mels=80, n_ceps=40, precise=True), 512, 64000)
    run("precise mode: default branch (MelSpectrogram + AmplitudeToDB), pad 16, 256 x 8 s", lid.FrontEnd(kind="melspec_db", pad=16, precise=True),
        256, 128000)
    run_resample("resample 44.1 kHz -> 16 kHz (475-tap polyphase FIR), 256 x 8 s", 44100, 256, 8.0)
    run_resample("resample 22.05 kHz -> 16 kHz (459-tap polyphase FIR), 256 x 8 s", 22050, 256, 8.0)
    run_resample("resample 25 kHz -> 16 kHz (45-tap polyphase FIR, 16 phases), 256 x 8 s", 25000, 256, 8.0)


def run_resample(name, orig, B, seconds, steps=None, warmup=5):
    if ONLY and ONLY not in name:
        return
    steps = steps or STEPS
    rs = lid.Resampler(orig, 16000)
    g = torch.Generator(device="cuda").manual_seed(2)
    n = int(orig * seconds)
    wavs = [torch.randn(n, device="cuda", generator=g) for _ in range(B)]
    for _ in range(warmup):
        rs.resample_list(wavs)
    # time the kernel itself: the list API concatenates its inputs first, which is not part of the resampling
    import ctypes as C
    packed = torch.cat(wavs)
    n_out = rs.out_len(n)
    stride = (n_out + 3) // 4 * 4
    out = torch.empty(B * stride, device="cuda")
    tab = torch.tensor([[i * n for i in range(B)], [n] * B, [i * stride for i in range(B)], [n_out] * B], dtype=torch.int64,
                       device="cuda")
    lib = lid.load_library()

    def launch():
        rc = lib.lidfe_resample(rs.handle, B, packed.data_ptr(), tab[0].data_ptr(), tab[1].data_ptr(), out.data_ptr(),
                                tab[2].data_ptr(), tab[3].data_ptr(), n_out, torch.cuda.current_stream().cuda_stream)
        assert rc == 0
    for _ in range(warmup):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    taps = rs.kernel.shape[1]
    print(json.dumps({"config": name, "utterances": B, "in_samples": n, "out_samples": n_out, "taps": taps,
                      "ms_per_step": round(ms, 5), "audio_s_per_s": round(B * seconds / (ms * 1e-3), 1),
                      "fp32_tflops": round(2.0 * B * n_out * taps / (ms * 1e-3) / 1e12, 2)}), flush=True)


if __name__ == "__main__":
    main()
