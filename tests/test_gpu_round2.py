"""Round-2 GPU tests: the warp-autonomous kernel against fbank_kernel, in-kernel Philox dither, the Kaldi window
selector, the fused normalize_wav load (featurize_raw), the plan pool, many short padded utterances (the arrival-counter
finding of ADVICE.md), the north-star multi-GPU path (cfg4) on 2 ranks over NCCL, and SURVEY.md 8(c)'s acceptance
metrics (ii) / (iv) in their UNRELAXED form as strict xfails (profiles/r2_parity_matrix.txt holds the counts).
Run on the B200 box: python -m pytest tests -m gpu."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import frontend_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------------
# Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11) restated in numpy --
# test infrastructure: the kernel's dither stream must be THIS function of (seed, utterance, sample)
# ---------------------------------------------------------------------------------------------------------------------
def philox4x32_10(ctr, key):
    """ctr: (..., 4) uint32, key: (2,) uint32 -> (..., 4) uint32"""
    c = [ctr[..., i].astype(np.uint64) for i in range(4)]
    k0, k1 = np.uint64(key[0]), np.uint64(key[1])
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c = [(hi1 ^ c[1] ^ k0) & mask, lo1, (hi0 ^ c[3] ^ k1) & mask, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & mask
        k1 = (k1 + np.uint64(0xBB67AE85)) & mask
    return np.stack(c, -1).astype(np.uint32)


def dither_uniform(seed, utt, n):
    """U[0,1) of samples 0..n-1 of utterance `utt` as the kernels draw it (lidfe_kernels.cuh: dither_uniform)."""
    blk = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.stack([blk & np.uint64(0xFFFFFFFF), blk >> np.uint64(32), np.full_like(blk, utt), np.zeros_like(blk)], -1).astype(np.uint32)
    r = philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)).reshape(-1)[:n]
    return ((r >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24))


def test_philox_known_answers():
    """Random123's published known-answer vectors for philox4x32-10 pin the numpy restatement (CPU)."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        got = philox4x32_10(np.array([ctr], dtype=np.uint32), key)[0]
        assert tuple(int(v) for v in got) == want


gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lid():
    import speech_lid_b200 as m
    return m


@pytest.fixture(scope="module")
def fe(lid):
    return lid.FrontEnd(n_mels=80)


def _fresh(ctor, env, *args, **kw):
    """An object created under temporary environment switches (they are read once, at creation)."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return ctor(*args, **kw)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _fresh_frontend(lid, env, **kw):
    """A FrontEnd created under temporary environment switches (they are read once, at lidfe_create)."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return lid.FrontEnd(**kw)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@gpu
def test_warp_kernel_equals_cta_kernel(lid):
    """The warp-autonomous kernel and fbank_kernel share their per-frame arithmetic: raw features are bit-equal on
    ragged padded / packed batches, float32 and int16 input, 80 and 40 mel bins; CMVN outputs agree to a few ulps (the
    statistics are summed in another order)."""
    g = torch.Generator().manual_seed(5)
    lens = [16000, 4000, 24000, 8560, 400, 559, 560, 64000, 1040, 720, 128000]
    for kw in (dict(), dict(in_dtype=torch.int16, in_scale=1.0 / 32768), dict(n_mels=40), dict(preemph=0.97, remove_dc=False)):
        fw = _fresh_frontend(lid, {"LIDFE_WARP_KERNEL": "1"}, **kw)
        fc = _fresh_frontend(lid, {"LIDFE_WARP_KERNEL": "0"}, **kw)
        if kw.get("in_dtype") == torch.int16:
            wavs = [(torch.randn(n, generator=g) * 3000).to(torch.int16) for n in lens]
        else:
            wavs = [torch.randn(n, generator=g) for n in lens]
        for padded in (True, False):
            pw, pc = fw.make_plan(lens, padded=padded), fc.make_plan(lens, padded=padded)
            packed = fw.pack(wavs, pw)
            a = fw.featurize_packed(packed, pw)
            b = fc.featurize_packed(packed, pc)
            assert torch.equal(a, b), (kw, padded)
            torch.manual_seed(3)
            masks = lid.draw_masks(pw.frames, fw.n_out, 0.05, 13, 2).cuda()
            assert torch.equal(fw.featurize_packed(packed, pw, masks=masks), fc.featurize_packed(packed, pc, masks=masks))
            ua = torch.nan_to_num(fw.featurize_packed(packed, pw, masks=masks, cmvn="utt"), nan=-7.0)
            ub = torch.nan_to_num(fc.featurize_packed(packed, pc, masks=masks, cmvn="utt"), nan=-7.0)
            assert torch.equal(ua == 0, ub == 0) and float((ua - ub).abs().max()) < 2e-6, (kw, padded)
            sa = torch.zeros(2 * fw.n_out + 1, dtype=torch.float64, device="cuda")
            sb = torch.zeros_like(sa)
            fw.featurize_packed(packed, pw, cmvn="global_accum", stats_out=sa)
            fc.featurize_packed(packed, pc, cmvn="global_accum", stats_out=sb)
            assert sa[-1] == sb[-1] == sum(pw.frames)
            assert float(((sa - sb).abs() / sb.abs().clamp_min(1.0)).max()) < 1e-7


@gpu
@pytest.mark.parametrize("pad", [0, 16])
def test_warp_kernel_equals_cta_kernel_default_branch(lid, pad):
    """The reference's default branch (MelSpectrogram + AmplitudeToDB(top_db=80), ref: lid/audio_processor.py:72-105) through
    the warp-autonomous kernel (CENTER framing: interior quads by TMA, the first quad and the last one or two of every
    utterance staged element by element with the reflection; per-utterance extrema by atomics) against fbank_kernel:
    same arithmetic per frame, max / min are order-free, so the outputs are bit-equal -- raw dB values, with masks, and after
    the top_db clamp -- on ragged padded / packed batches including utterances that are edge from end to end, with a
    quiet tail that the clamp actually touches, over repeated launches (launch parity of the extrema workspace)."""
    g = torch.Generator().manual_seed(50 + pad)
    lens = [16000, 4000, 24000, 8560, 400, 559, 257, 64000, 1040, 720, 128000, 300, 880, 881]
    wavs = [torch.randn(n, generator=g) for n in lens]
    wavs[3][4000:] *= 1e-5                      # 100 dB down: AmplitudeToDB's clamp is active there
    wavs[10][96000:] *= 1e-6
    fw = _fresh_frontend(lid, {"LIDFE_WARP_KERNEL": "1"}, kind="melspec_db", pad=pad)
    fc = _fresh_frontend(lid, {"LIDFE_WARP_KERNEL": "0"}, kind="melspec_db", pad=pad)
    for padded in (True, False):
        pw, pc = fw.make_plan(lens, padded=padded), fc.make_plan(lens, padded=padded)
        assert pw.frames == pc.frames == [1 + (n + 2 * pad) // 160 for n in lens]
        packed = fw.pack(wavs, pw)
        torch.manual_seed(3)
        masks = lid.draw_masks(pw.frames, 80, 0.05, 27, 2).cuda()
        for rep in range(3):
            a = fw.featurize_packed(packed, pw, masks=masks if rep % 2 else None)
            b = fc.featurize_packed(packed, pc, masks=masks if rep % 2 else None)
            assert torch.equal(a, b), (pad, padded, rep)
            assert bool(torch.isfinite(a).all())
    # and against the oracle on one utterance with a clamped tail
    want = O.melspec_db(wavs[3].unsqueeze(0), pad=pad)[0].T
    got = fw.featurize([wavs[3]])[0][0].cpu()
    assert got.shape == want.shape
    assert float((got - want).abs().max() / want.abs().max()) <= 1e-4


@gpu
def test_many_short_utterances_padded_equals_packed(lid):
    """ADVICE.md (round 1): a padded batch of many short utterances with cmvn='none' (zero-fill work between real work)
    must give the packed layout's bits, row for row, launch after launch."""
    g = torch.Generator().manual_seed(77)
    lens = torch.randint(400, 4000, (600,), generator=g).tolist()
    wavs = [torch.randn(n, generator=g) for n in lens]
    for env in ({"LIDFE_WARP_KERNEL": "1"}, {"LIDFE_WARP_KERNEL": "0"}):
        f = _fresh_frontend(lid, env)
        pp, pk = f.make_plan(lens, padded=True), f.make_plan(lens, padded=False)
        packed = f.pack(wavs, pp)
        ref = f.featurize_packed(packed, pk).cpu()
        for _ in range(4):
            out = f.featurize_packed(packed, pp).cpu()
            row = 0
            for i, T in enumerate(pp.frames):
                assert torch.equal(out[i, :T], ref[row:row + T]), (env, i)
                assert torch.all(out[i, T:] == 0)
                row += T


@gpu
def test_inkernel_dither_is_the_philox_stream(lid):
    """NS1: cfg.dither > 0 adds dither * U[0,1) inside the fused kernel, U = Philox4x32-10 keyed by (seed, utterance,
    sample) -- no host-drawn noise crosses PCIe.  (ref: lid/audio_processor.py:129 draws torch.rand_like on the host;
    its kaldi call passes dither=0.0, :57.)  The device draw must be the published Philox function, the features must be
    the oracle's features of (wav + dither * U), and another seed must give another stream."""
    seed, amp = 0x1234567811, 0.05
    lens = [16000, 4803, 9000]
    wavs = [O.synth_noise(n, 900 + i) for i, n in enumerate(lens)]
    f0 = lid.FrontEnd()
    plan = f0.make_plan(lens, padded=False)
    zeros = torch.zeros(plan.total_samples, device="cuda")
    fd = lid.FrontEnd(dither=amp, seed=seed)
    pd = fd.make_plan(lens, padded=False)
    u_dev = fd.wave_stages(zeros, pd, dither=1.0).cpu()           # 0 + 1.0 * U: the device's draw
    for i, (o, n) in enumerate(zip(pd.offsets, lens)):
        u = dither_uniform(seed, i, n)
        assert np.array_equal(u_dev[o:o + n].numpy(), u), "utterance %d: device draw != Philox4x32-10" % i
        assert abs(float(u.mean()) - 0.5) < 0.02 and u.min() >= 0.0 and u.max() < 1.0
        hist = np.histogram(u, bins=10, range=(0, 1))[0] / n
        assert np.abs(hist - 0.1).max() < 0.02
    got = fd.featurize_packed(fd.pack(wavs, pd), pd).cpu()
    again = fd.featurize_packed(fd.pack(wavs, pd), pd).cpu()
    assert torch.equal(got, again)                                 # counter based: no state between launches
    row = 0
    for i, w in enumerate(wavs):
        noisy = w + np.float32(amp) * torch.from_numpy(dither_uniform(seed, i, lens[i])).unsqueeze(0)
        want = O.kaldi_fbank(noisy)
        err = float((got[row:row + want.shape[0]] - want).abs().max() / want.abs().max())
        assert err <= 3e-4, (i, err)
        row += want.shape[0]
    other = lid.FrontEnd(dither=amp, seed=seed + 1)
    po = other.make_plan(lens, padded=False)
    assert not torch.equal(other.featurize_packed(other.pack(wavs, po), po).cpu(), got)
    plain = f0.featurize_packed(f0.pack(wavs, plan), plan).cpu()
    assert not torch.equal(plain, got)


@gpu
@pytest.mark.parametrize("window", ["hamming", "hanning", "rectangular", "blackman", "povey"])
def test_kaldi_window_types(lid, window):
    """NS1: the window selector (ta: compliance/kaldi.py:86-113), each against the oracle (pinned bit-exact against
    torchaudio in tests/test_oracle_golden.py)."""
    f = lid.FrontEnd(window=window)
    wavs = [O.synth_speechlike(24000, 31), O.synth_noise(16000, 32)]
    feats, _ = f.featurize(wavs)
    feats = feats.cpu()
    for i, w in enumerate(wavs):
        want = O.kaldi_fbank(w, window_type=window)
        got = feats[i, :want.shape[0]]
        tol = 1e-4 if i == 0 else 3e-4          # white noise: the cancellation-dominated low bins (see test_gpu_parity.py)
        assert float((got - want).abs().max() / want.abs().max()) <= tol, (window, i)
    with pytest.raises(Exception):
        lid.FrontEnd(window="kaiser")


@gpu
def test_featurize_raw_fused_normalize(lid):
    """Row f2: int16 PCM in, normalize_wav applied while the kernel stages the samples (statistics pre-pass + ONE fused
    kernel).  Same bits as wave_stages (normalise, write fp32) followed by the plain kernel; parity with the oracle chain
    read_audio(normalize=True) -> wav2mel (ref: lid/audio_processor.py:108-122, :41-69)."""
    g = torch.Generator().manual_seed(21)
    lens = [16000, 23456, 9000, 40000, 801]
    pcm = [(torch.randn(n, generator=g) * 2500 + 30).clamp(-32768, 32767).to(torch.int16) for n in lens]
    f16 = lid.FrontEnd(in_dtype=torch.int16, in_scale=1.0 / 32768.0)
    f32 = lid.FrontEnd()
    p16 = f16.make_plan(lens, padded=True)
    p32 = f32.make_plan(lens, padded=True, offsets=p16.offsets)
    packed = f16.pack(pcm, p16)
    fused = f16.featurize_packed(packed, p16, raw=True)
    two = f32.featurize_packed(f32.wave_stages(packed, p32, normalize=True), p32)
    assert torch.equal(fused, two)
    for i, w in enumerate(pcm):
        want = O.kaldi_fbank(O.normalize_wav(w.float().unsqueeze(0) * (1.0 / 32768.0)))
        got = fused[i, :want.shape[0]].cpu()
        assert float((got - want).abs().max() / want.abs().max()) <= 3e-4, i


@gpu
def test_s3prl_fbank_variant_matches_reference_module(lid):
    """Row f4: speech_lid_b200.S3prlFBank (windowed-DFT GEMM on the tensor cores + mel / dB / scalar normalisation)
    against outputs of the reference's own FBank class (ref: wav2vec-exp/s3prl_model.py:174-204) and, on a ragged batch,
    against the oracle.  Tolerance: 1e-4 of the feature range (the values are (x - mean) / std of a dB spectrogram)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "s3prl_fbank.npz"))
    mods = {}
    for k in "abcde":
        n_fft = int(z["nfft_" + k])
        fb = mods.setdefault(n_fft, lid.S3prlFBank(80, n_fft))
        x = torch.from_numpy(z["in_" + k]).reshape(-1)
        want = torch.from_numpy(z["out_" + k])
        got = fb(x)
        assert got.shape == want.shape and got.device.type == "cpu", (k, got.shape, want.shape)
        if want.shape[-1] > 1:
            assert float((got - want).abs().max() / want.abs().max()) <= 1e-4, k
        assert fb(x.cuda()).is_cuda
    g = torch.Generator().manual_seed(4)
    wavs = [torch.randn(n, generator=g) for n in (640, 641, 16000, 40017, 959, 128 * 320 + 640, 3200)]
    fb = mods[640]
    outs = fb.forward_list([w.cuda() for w in wavs])
    raw = fb.forward_list([w.cuda() for w in wavs], normalize=False)
    for w, o, r in zip(wavs, outs, raw):
        want = O.s3prl_fbank(w, 80, 640)[0].T if O.s3prl_fbank(w, 80, 640).dim() == 3 else O.s3prl_fbank(w, 80, 640).T
        want_raw = O.s3prl_fbank(w, 80, 640, normalize=False)
        want_raw = (want_raw[0] if want_raw.dim() == 3 else want_raw).T
        assert o.shape == want.shape == (fb.num_frames(w.numel()), 80)
        assert float((r.cpu() - want_raw).abs().max() / want_raw.abs().max()) <= 1e-4, w.numel()
        assert float((o.cpu() - want).abs().max() / want.abs().max()) <= 1e-4, w.numel()
    with pytest.raises(RuntimeError):
        fb.forward_list([torch.randn(639)])


def _cuda_kernels(fn):
    """Names of the CUDA kernels that fn() launches (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


@gpu
@pytest.mark.parametrize("orig", [44100, 22050, 25000, 15000])
def test_resampler_kernels_agree_tcgen05_fp32(lid, orig):
    """Row f4: the two kernels behind lidfe_resample -- resample_tc_kernel (tcgen05 + TMEM, 3 x TF32, what a Resampler
    runs on sm_100 whenever the reduced output rate is a multiple of 16) and the FP32 resample_kernel -- against an fp64
    evaluation of the same polyphase sum with the same fp32 FIR bank (ta: functional/functional.py
    _apply_sinc_resample_kernel), on ragged utterances: shorter than one tile, one sample, exact multiples of the period,
    several 128-frame tiles (the persistent CTA walks them through both TMEM accumulator buffers and wraps the 3-stage
    pipeline many times).  25 kHz has 16 phases (one 16-column phase tile), 15 kHz 29 taps (a second, all-zero tap
    block)."""
    import math
    g = torch.Generator().manual_seed(orig)
    lens = [int(orig * s) for s in (0.05, 0.31, 1.0, 2.57, 0.011, 6.3)] + [441, 1, 44101, 441 * 128, 441 * 128 + 1]
    wavs = [torch.randn(n, generator=g) for n in lens]
    outs = {}
    for kind, kernel in (("tc", "resample_tc_kernel"), ("fp32", "resample_kernel")):
        rs = lid.Resampler(orig, 16000) if kind == "tc" else _fresh(lid.Resampler, {"LIDFE_RESAMPLE_TC": "0"}, orig, 16000)
        gg = math.gcd(rs.orig_freq, rs.new_freq)
        o_red = rs.orig_freq // gg
        k64 = rs.kernel.double()
        dev = [w.cuda() for w in wavs]
        res, names = _cuda_kernels(lambda: rs.resample_list(dev))
        ran_tc = any("resample_tc_kernel" in n for n in names)
        assert ran_tc == (kind == "tc") and any(kernel in n for n in names), (kind, names)
        for w, o in zip(wavs, res):
            x = torch.nn.functional.pad(w.double(), (rs.width, rs.width + o_red))
            want = (x.unfold(0, k64.shape[1], o_red) @ k64.T).reshape(-1)[:rs.out_len(w.numel())]
            assert o.numel() == want.numel(), (kind, w.numel())
            assert float((o.double().cpu() - want).abs().max()) <= 1e-5, (kind, w.numel())
        outs[kind] = [o.cpu() for o in res]
    worst = max(float((a - b).abs().max()) for a, b in zip(outs["tc"], outs["fp32"]))
    assert worst <= 2e-6, worst


@gpu
@pytest.mark.parametrize("in_dtype", [torch.float32, torch.int16])
def test_pack_paths_agree(lid, in_dtype):
    """FrontEnd.pack: pageable sources (native threaded packer -> pinned staging, shipped in groups), pinned sources
    (lidfe_h2d_gather, no staging) and device sources give the same packed buffer, gaps zero; repeated calls re-use the
    two staging buffers without tearing (the ragged collate path, ref: lid/raw_datasets.py:345-351)."""
    kw = dict(in_dtype=torch.int16, in_scale=1.0 / 32768) if in_dtype == torch.int16 else {}
    f = lid.FrontEnd(**kw)
    g = torch.Generator().manual_seed(21)
    for rep, B in enumerate((3, 40, 200)):
        lens = torch.randint(400, 200000 if B < 100 else 120000, (B,), generator=g).tolist()
        wavs = [(torch.randn(n, generator=g) * 2000).to(in_dtype) for n in lens]
        plan = f.make_plan(lens, padded=True)
        want = torch.zeros(plan.total_samples, dtype=in_dtype)
        for w, o, n in zip(wavs, plan.offsets, plan.lengths):
            want[o:o + n] = w
        a = f.pack(wavs, plan)
        b = f.pack([w.pin_memory() for w in wavs], plan)
        c = f.pack([w.cuda() for w in wavs], plan)
        d = f.pack([w.unsqueeze(0) for w in wavs], plan)                  # (1, N): channel 0
        torch.cuda.synchronize()
        for name, got in (("pageable", a), ("pinned", b), ("device", c), ("2-d", d)):
            assert torch.equal(got.cpu(), want), (name, rep)
        plan.close()


@gpu
def test_plan_pool_serves_ragged_batches_without_allocating(lid):
    """VERDICT r1 #7: a new length signature every step (ref: lid/raw_datasets.py:345-365) must not allocate once the
    pool is warm: plans take their device / pinned memory from the handle's pool."""
    f = lid.FrontEnd()
    g = torch.Generator().manual_seed(9)
    collate = lid.DeviceCollate(f, {"a": 0}, train=True, cmvn="utt")

    def batch():
        lens = torch.randint(8000, 48000, (24,), generator=g).tolist()
        return [(torch.randn(n, generator=g), torch.zeros(3, dtype=torch.long), "p", "a") for n in lens]

    for _ in range(6):
        collate(batch())
    torch.cuda.synchronize()
    allocated, _ = f.pool_stats()
    for _ in range(12):
        feats = collate(batch())[0]
        assert torch.isfinite(feats).all()
    torch.cuda.synchronize()
    assert f.pool_stats()[0] == allocated, "plan pool grew in steady state"


# ---------------------------------------------------------------------------------------------------------------------
# cfg4 on two ranks over NCCL
# ---------------------------------------------------------------------------------------------------------------------
_CFG4_WORKER = r"""
import os, sys, torch
sys.path.insert(0, {root!r})
import torch.distributed as dist
import speech_lid_b200 as lid
from oracle import frontend_oracle as O
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
g = torch.Generator().manual_seed(3)
lengths = torch.randint(16000, 160001, (24,), generator=g).tolist()
shards = lid.lpt_partition(lengths, world)
fe = lid.FrontEnd(device="cuda:%d" % rank)
mine = shards[rank]
wavs = [O.synth_noise(lengths[i], 700 + i) for i in mine]
plan = fe.make_plan([lengths[i] for i in mine], padded=False)
packed = fe.pack(wavs, plan)
torch.manual_seed(5 + rank)
masks = lid.draw_masks(plan.frames, 80, 0.05, 27, 2).cuda()
stats = torch.zeros(161, dtype=torch.float64, device="cuda")
out = fe.featurize_packed(packed, plan, cmvn="global_accum", stats_out=stats)
raw = out.clone()
lid.allreduce_stats(stats)                      # the one collective of the path: 161 doubles over NCCL
fe.cmvn_apply(out, plan, stats, masks=masks)
torch.cuda.synchronize()
torch.save(dict(stats=stats.cpu(), out=out.cpu(), raw=raw.cpu(), mine=mine, frames=plan.frames, masks=masks.cpu(), lengths=lengths),
           os.path.join({out!r}, "rank%d.pt" % rank))
dist.destroy_process_group()
"""


@gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_cfg4_global_cmvn_two_ranks_nccl(tmp_path):
    """North-star multi-GPU path (SURVEY.md 8e, BASELINE cfg4): ragged utterances, LPT shard by utterance, packed
    featurize with statistics, ONE all_reduce(161 fp64) over NCCL, normalise + mask.  Checked against the oracle chain
    over the whole (unsharded) set."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "worker.py"
    script.write_text(_CFG4_WORKER.format(root=ROOT, out=str(tmp_path)))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env))
    for p in procs:
        assert p.wait(timeout=600) == 0
    d = [torch.load(os.path.join(str(tmp_path), "rank%d.pt" % r)) for r in range(2)]
    lengths = d[0]["lengths"]
    assert sorted(d[0]["mine"] + d[1]["mine"]) == list(range(len(lengths)))            # every utterance on exactly one rank
    feats = {}
    for r in range(2):
        row = 0
        for i, T in zip(d[r]["mine"], d[r]["frames"]):
            feats[i] = (r, row, T)
            row += T
    # the all-reduced sums equal the sums over every rank's raw rows (and both ranks hold the same vector)
    allraw = torch.cat([d[r]["raw"] for r in range(2)]).double()
    want_stats = torch.cat([allraw.sum(0), (allraw * allraw).sum(0), torch.tensor([float(allraw.shape[0])], dtype=torch.float64)])
    for r in range(2):
        assert torch.allclose(d[r]["stats"], want_stats, rtol=1e-7, atol=1e-6)
    assert torch.equal(d[0]["stats"], d[1]["stats"])
    mean, std = allraw.mean(0), allraw.std(0, unbiased=True)
    for i, (r, row, T) in feats.items():
        k = d[r]["mine"].index(i)
        b = [tuple(int(v) for v in d[r]["masks"][k, q]) for q in range(2)]
        # the device's arithmetic on its own raw rows (tight) ...
        ref = ((d[r]["raw"][row:row + T].double() - mean) / (std + 1e-9)).float()
        ref = O.apply_mask_bounds(ref.T.unsqueeze(0), b)[0].T
        got = d[r]["out"][row:row + T]
        assert torch.allclose(got, ref, rtol=1e-5, atol=1e-5), i
        assert torch.equal(got == 0, ref == 0)
        # ... and the raw rows against the oracle's fbank of the same utterance
        want = O.kaldi_fbank(O.synth_noise(lengths[i], 700 + i))
        assert float((d[r]["raw"][row:row + T] - want).abs().max() / want.abs().max()) <= 3e-4


# ---------------------------------------------------------------------------------------------------------------------
# SURVEY.md 8(c) metrics (ii) and (iv) exactly as written -- strict xfails, so the gap stays visible.
# profiles/r2_parity_matrix.txt: pass / fail counts for every BASELINE config, next to an independent CPU fp32 library
# under the same rule.
# ---------------------------------------------------------------------------------------------------------------------
def _strict_inputs():
    return [O.synth_noise(128000, 100 + s) for s in range(16)]


@gpu
@pytest.mark.xfail(strict=True, reason="(ii) over ALL bins on white noise: the reference's own fp32 error against fp64 reaches "
                   "1e-4 of the range in mel bins 0-2 (pre-emphasis 1.0 leaves them cancellation dominated), so no second fp32 "
                   "pipeline -- numpy's pocketfft on the reference's own frames included -- stays within 1e-4 of it on every "
                   "utterance; see profiles/r2_parity_matrix.txt")
def test_strict_metric_ii_all_bins_white_noise(fe):
    wavs = _strict_inputs()
    feats, _ = fe.featurize(wavs)
    feats = feats.cpu()
    for i, w in enumerate(wavs):
        want = O.kaldi_fbank(w)
        assert float((feats[i, :want.shape[0]] - want).abs().max() / want.abs().max()) <= 1e-4


@gpu
@pytest.mark.xfail(strict=True, reason="(iv) per mel bin, max over frames, <= 1.5 x the reference's own error against fp64: the "
                   "maximum over ~800 frames of a heavy-tailed error is decided by single frames; the kernel's 16 x 16 FFT with "
                   "its real-FFT split carries a somewhat higher round-off floor than MKL's real FFT; see "
                   "profiles/r2_parity_matrix.txt for the counts")
def test_strict_metric_iv_per_bin_white_noise(fe):
    wavs = _strict_inputs()
    feats, _ = fe.featurize(wavs)
    feats = feats.cpu()
    for i, w in enumerate(wavs):
        ref, tru = O.kaldi_fbank(w), O.truth64_fbank(w)
        eg = (feats[i, :ref.shape[0]].double() - tru).abs().max(0).values
        er = (ref.double() - tru).abs().max(0).values
        assert bool((eg <= 1.5 * er).all())


# ---------------------------------------------------------------------------------------------------------------------
# cfg5: the reference's Conformer consumer on the device (row A10)
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "lid", "ConformerLangModel.py")),
                    reason="baseline/_ref/lid not staged (__graft_entry__.build() copies it where /root/reference exists)")
def test_cfg5_reference_consumer_on_device():
    """On-device features -> the reference's ConformerMutiLangModel forward on the GPU (random init, eval, lang=None;
    ref: lid/ConformerLangModel.py:77-83, :272-294): CTC logits and language-id scores from the kernel's features equal
    those from the oracle's features (the reference's arithmetic) to well under the spread between classes."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import cfg5_device
    r = cfg5_device.run(B=16, n_check=8, steps=1)
    assert r is not None
    assert r["features_norm_rel_vs_oracle"] <= 3e-4
    assert r["consumer_worst_abs_diff"] <= 1e-3, r["consumer"]
    assert r["consumer_min_argmax_agreement"] >= 0.995, r["consumer"]
    assert 0.0 < r["frontend_share"] < 1.0


@gpu
def test_cfg5_conformer_consumer_on_device():
    """Row A10 where the reference's model source is not staged: the same consumer check through a stand-in Conformer of
    the reference model's shape (tools/cfg5_device.stand_in_model: torchaudio.models.Conformer, random init, eval).  The
    oracle's features are pinned to the reference's own outputs (tests/golden/), so this still compares the kernel with
    the reference's arithmetic as seen by a Conformer consumer; the convolutions run in plain fp32 (no TF32), so that
    only the two feature sets differ."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import cfg5_device
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        r = cfg5_device.run(B=16, n_check=8, steps=1, model=cfg5_device.stand_in_model())
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    assert r["features_norm_rel_vs_oracle"] <= 3e-4
    assert r["consumer_worst_abs_diff"] <= 1e-3, r["consumer"]
    assert r["consumer_min_argmax_agreement"] >= 0.995, r["consumer"]
    assert 0.0 < r["frontend_share"] < 1.0
