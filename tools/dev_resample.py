#!/usr/bin/env python
"""Development: the two resampler kernels (tcgen05 / FP32, selected by LIDFE_RESAMPLE_TC at Resampler creation) against an fp64 evaluation of the same polyphase sum, on ragged batches, and their timings on
256 x 8 s.  Run under `timeout`."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import speech_lid_b200 as lid


def make(kind, orig):
    os.environ["LIDFE_RESAMPLE_TC"] = "1" if kind == "tc" else "0"
    return lid.Resampler(orig, 16000)


def truth(rs, w):
    """fp64 polyphase sum with the same fp32 FIR bank (ta: functional/functional.py _apply_sinc_resample_kernel)."""
    import math
    g = math.gcd(rs.orig_freq, rs.new_freq)
    orig, new = rs.orig_freq // g, rs.new_freq // g
    k = rs.kernel.double()                                     # [new, taps]
    x = torch.nn.functional.pad(w.double().cpu(), (rs.width, rs.width + orig))
    fr = x.unfold(0, k.shape[1], orig)                         # [frames, taps]
    y = (fr @ k.T).reshape(-1)
    return y[:rs.out_len(w.numel())]


CHECK = os.environ.get("DEV_RS_NOCHECK") is None
for orig in ((44100, 22050) if CHECK else ()):
    g = torch.Generator().manual_seed(orig)
    lens = [int(orig * s) for s in (0.05, 0.31, 1.0, 2.57, 0.011)] + [441, 1, 44101]
    wavs = [torch.randn(n, generator=g) for n in lens]
    ref = None
    for kind in ("tc", "fp32"):
        rs = make(kind, orig)
        outs = rs.resample_list([w.cuda() for w in wavs])
        torch.cuda.synchronize()
        worst = 0.0
        for w, o in zip(wavs, outs):
            t = truth(rs, w)
            assert o.numel() == t.numel(), (kind, o.numel(), t.numel())
            worst = max(worst, float((o.double().cpu() - t).abs().max()))
        print("%d Hz %-5s max|err| vs fp64 %.3g" % (orig, kind, worst), flush=True)
        assert worst < 2e-5, (orig, kind, worst)

B, seconds = 256, 8.0
for orig in (44100, 22050):
    n = int(orig * seconds)
    gg = torch.Generator(device="cuda").manual_seed(2)
    packed = torch.randn(B * n, device="cuda", generator=gg)
    for kind in ("tc", "fp32"):
        rs = make(kind, orig)
        n_out = rs.out_len(n)
        stride = (n_out + 3) // 4 * 4
        out = torch.empty(B * stride, device="cuda")
        tab = torch.tensor([[i * n for i in range(B)], [n] * B, [i * stride for i in range(B)], [n_out] * B], dtype=torch.int64, device="cuda")
        lib = lid.load_library()

        def launch():
            rc = lib.lidfe_resample(rs.handle, B, packed.data_ptr(), tab[0].data_ptr(), tab[1].data_ptr(), out.data_ptr(),
                                    tab[2].data_ptr(), tab[3].data_ptr(), n_out, torch.cuda.current_stream().cuda_stream)
            assert rc == 0
        for _ in range(5):
            launch()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(30):
            launch()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 30
        taps = rs.kernel.shape[1]
        print("%d Hz %-5s %.3f ms  %.2f M audio-s/s  %.1f TFLOP/s (fp32-equivalent 2*taps per output sample)" % (
            orig, kind, ms, B * seconds / ms / 1e3, 2.0 * B * n_out * taps / (ms * 1e-3) / 1e12), flush=True)
