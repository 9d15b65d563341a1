"""Additive noise at a per-utterance SNR (noise.py, FrontEnd.add_noise, lidfe_add_noise): the host draw and its
validation and the numpy restatement of the Gaussian stream on the CPU; the device mix against
torchaudio.functional.add_noise, its special cases, the end-to-end and DeviceCollate paths on the GPU."""
import math

import numpy as np
import pytest
import torch
from scipy import stats

import speech_lid_b200 as lid
from speech_lid_b200.noise import NoiseDraw, noise_table
from oracle import frontend_oracle as O

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# Philox4x32-10 restated in numpy (the same function as tests/test_gpu_round2.py, pinned there by Random123's
# known-answer vectors) and the Box-Muller stream of lidfe_kernels.cuh: gauss_noise
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


def gauss_noise(seed, utt, n):
    """N(0,1) of samples 0..n-1 of utterance `utt` in fp64: counter (i >> 2, utt, 1), Box-Muller on (x, y), (z, w)."""
    blk = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.stack([blk & np.uint64(0xFFFFFFFF), blk >> np.uint64(32), np.full_like(blk, utt), np.ones_like(blk)], -1).astype(np.uint32)
    r = philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)).astype(np.float64)
    r = np.floor(r / 256.0)
    u1 = (r[:, 0::2] + 1.0) * 2.0 ** -24
    u2 = r[:, 1::2] * 2.0 ** -24
    rad = np.sqrt(-2.0 * np.log(u1))
    c, s = rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)
    return np.stack([c[:, 0], s[:, 0], c[:, 1], s[:, 1]], -1).reshape(-1)[:n]


def test_gauss_stream_is_normal():
    z = gauss_noise(0x5EED1234ABCD, 3, 1 << 20)
    assert abs(z.mean()) < 5e-3 and abs(z.var() - 1.0) < 5e-3
    assert stats.kstest(z, "norm").pvalue > 1e-3
    assert not np.array_equal(z[:1000], gauss_noise(0x5EED1234ABCD, 4, 1000))


# ---------------------------------------------------------------------------------------------------------------------
# host side (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def _cpu_bank(lengths=(5, 300, 17)):
    return lid.NoiseBank([torch.randn(n, generator=torch.Generator().manual_seed(n)) for n in lengths], device="cpu")


def test_draw_noise_known_answer():
    """The documented draw order, pinned: keep uniforms, SNR uniforms, clip indices, start uniforms, seed."""
    bank = _cpu_bank()
    assert bank.offsets == [0, 5, 305] and bank.lengths == [5, 300, 17] and bank.data.numel() == 322
    d = lid.draw_noise(6, (-5.0, 20.0), p=0.5, bank=bank, generator=torch.Generator().manual_seed(7))
    assert d.snr_db.dtype == torch.float32
    assert d.snr_db.tolist() == [2.367802619934082, 9.01803970336914, math.inf, math.inf, math.inf, math.inf]
    assert d.clip.tolist() == [1, 2, 2, 1, 0, 2] and d.start.tolist() == [254, 0, 16, 32, 4, 15]
    assert d.seed == 8303423580812505379
    g = lid.draw_noise(3, 10.0, generator=torch.Generator().manual_seed(1234))
    assert g.snr_db.tolist() == [10.0] * 3 and g.clip is None and g.start is None and g.seed == 5099865445391015966
    # ranges: SNR in [lo, hi), starts inside their clips
    d = lid.draw_noise(4000, (3.0, 7.5), bank=bank, generator=torch.Generator().manual_seed(1))
    assert float(d.snr_db.min()) >= 3.0 and float(d.snr_db.max()) <= 7.5
    lens = torch.tensor(bank.lengths)[d.clip]
    assert bool((d.start >= 0).all()) and bool((d.start < lens).all()) and set(d.clip.tolist()) == {0, 1, 2}
    tab, snr = noise_table(d, bank, 4000)
    assert tab.shape == (3, 4000) and torch.equal(tab[1], lens) and torch.equal(tab[2], d.start)
    assert torch.equal(tab[0], torch.tensor(bank.offsets)[d.clip]) and torch.equal(snr, d.snr_db)


def test_draw_noise_p0_is_all_clean():
    d = lid.draw_noise(50, (0.0, 20.0), p=0.0, generator=torch.Generator().manual_seed(3))
    assert bool(torch.isinf(d.snr_db).all()) and bool((d.snr_db > 0).all())
    # the stream advances by the same amount whatever p is
    g0, g1 = torch.Generator().manual_seed(3), torch.Generator().manual_seed(3)
    lid.draw_noise(50, (0.0, 20.0), p=0.0, generator=g0)
    lid.draw_noise(50, (0.0, 20.0), p=1.0, generator=g1)
    assert torch.equal(torch.rand(4, generator=g0), torch.rand(4, generator=g1))


def test_noise_validation():
    with pytest.raises(ValueError):
        lid.NoiseBank([], device="cpu")
    with pytest.raises(ValueError, match="empty"):
        lid.NoiseBank([torch.randn(10), torch.zeros(0)], device="cpu")
    with pytest.raises(ValueError, match="zero energy"):
        lid.NoiseBank([torch.zeros(100)], device="cpu")
    with pytest.raises(ValueError, match="non-finite"):
        lid.NoiseBank([torch.tensor([1.0, float("nan")])], device="cpu")
    for bad in (float("nan"), -math.inf, (5.0, 1.0), (0.0, math.inf), (float("nan"), 1.0)):
        with pytest.raises(ValueError):
            lid.draw_noise(4, bad)
        with pytest.raises(ValueError):
            lid.NoiseAugment(None, bad)
    for p in (-0.1, 1.5):
        with pytest.raises(ValueError):
            lid.draw_noise(4, 10.0, p=p)
    assert bool(torch.isinf(lid.draw_noise(2, math.inf).snr_db).all())        # a number +inf: all clean
    bank = _cpu_bank()
    ok = NoiseDraw(snr_db=torch.tensor([1.0, 2.0]), clip=torch.tensor([0, 2]), start=torch.tensor([4, 16]), seed=0)
    noise_table(ok, bank, 2)
    for kw, msg in ((dict(clip=torch.tensor([0, 3])), "clip"), (dict(clip=torch.tensor([-1, 0])), "clip"),
                    (dict(start=torch.tensor([5, 0])), "start"), (dict(start=torch.tensor([0, -1])), "start"),
                    (dict(snr_db=torch.tensor([float("nan"), 1.0])), "NaN"),
                    (dict(snr_db=torch.tensor([-math.inf, 1.0])), "NaN"), (dict(clip=None), "bank")):
        d = NoiseDraw(**{**ok.__dict__, **kw})
        with pytest.raises(ValueError, match=msg):
            noise_table(d, bank, 2)
    with pytest.raises(ValueError):
        noise_table(ok, bank, 3)


# ---------------------------------------------------------------------------------------------------------------------
# device (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _bits(t):
    return t.contiguous().view(torch.int32)


def _window(clip, start, n):
    """nu = clip[(start + i) mod len(clip)], i < n: the looped segment, built on the host"""
    idx = (start + np.arange(n)) % clip.numel()
    return clip[torch.from_numpy(idx)]


def _add_noise64(x, nu, snr):
    """torchaudio.functional.add_noise in fp64 on the fp32 x and nu, and its gain"""
    import torchaudio.functional as F
    x64, nu64 = x.double(), nu.double()
    y = F.add_noise(x64.unsqueeze(0), nu64.unsqueeze(0), torch.tensor([float(snr)], dtype=torch.float64))[0]
    a = math.sqrt(float((x64 ** 2).sum()) / float((nu64 ** 2).sum()) * 10.0 ** (-float(snr) / 10.0))
    return y, a


@pytest.fixture(scope="module")
def fe():
    return lid.FrontEnd(n_mels=80)


@gpu
@pytest.mark.parametrize("i16", [False, True])
def test_bank_noise_matches_torchaudio(fe, i16):
    """Ragged batch, unaligned packing, clips shorter than their utterance (wrap), starts near the clip's end, odd
    clip offsets in the bank: every sample within 2^-22 (|x| + |a nu|) of torchaudio's fp64 mix, the realised SNR
    within 1e-3 dB."""
    g = torch.Generator().manual_seed(21)
    lens = [16000, 7001, 3333, 24000, 9999]
    clips = [torch.randn(n, generator=g) * s for n, s in ((5003, 0.3), (20001, 1.0), (997, 2.0), (40000, 0.05))]
    bank = lid.NoiseBank(clips)
    offsets, pos = [], 3
    for n in lens:
        offsets.append(pos)
        pos += n + 5                                       # nothing 16-byte aligned
    plan = fe.make_plan(lens, padded=False, offsets=offsets)
    if i16:
        pcm = [(torch.randn(n, generator=g) * 4000).to(torch.int16) for n in lens]
        xs = [p.to(torch.float32) * np.float32(1.0 / 32768) for p in pcm]
        packed = torch.zeros(pos + 7, dtype=torch.int16)
        for o, p in zip(offsets, pcm):
            packed[o:o + p.numel()] = p
    else:
        xs = [torch.randn(n, generator=g) * (0.1 + i) for i, n in enumerate(lens)]
        packed = torch.zeros(pos + 7)
        for o, x in zip(offsets, xs):
            packed[o:o + x.numel()] = x
    clip = torch.tensor([0, 2, 2, 1, 3])
    start = torch.tensor([5000, 996, 10, 19990, 123])      # near the end: the window wraps at once
    snr = torch.tensor([-5.0, 0.0, 17.5, 40.0, 9.25])
    draw = NoiseDraw(snr_db=snr, clip=clip, start=start, seed=0)
    y = fe.add_noise(packed.cuda(), plan, draw, bank=bank).cpu()
    gaps = torch.ones(y.numel(), dtype=torch.bool)
    for i, (o, n) in enumerate(zip(offsets, lens)):
        gaps[o:o + n] = False
        x = xs[i]
        nu = _window(clips[int(clip[i])], int(start[i]), n)
        y64, a = _add_noise64(x, nu, float(snr[i]))
        got = y[o:o + n].double()
        bound = 2.0 ** -22 * (x.double().abs() + a * nu.double().abs())
        assert bool(((got - y64).abs() <= bound).all()), (i, float(((got - y64).abs() / bound).max()))
        d = got - x.double()
        realised = 10 * math.log10(float((x.double() ** 2).sum()) / float((d ** 2).sum()))
        assert abs(realised - float(snr[i])) <= 1e-3, (i, realised)
    assert bool((y[gaps] == 0).all())


@gpu
def test_gaussian_noise_is_the_philox_stream(fe):
    lens = [50000, 1237, 20480]
    plan = fe.make_plan(lens, padded=False)
    ones = torch.ones(plan.total_samples, device="cuda")
    seed = 0x0123456789ABCDEF
    draw = NoiseDraw(snr_db=torch.full((3,), -40.0), clip=None, start=None, seed=seed)
    y = fe.add_noise(ones, plan, draw)
    again = fe.add_noise(ones, plan, draw)
    assert torch.equal(_bits(y), _bits(again))
    other = fe.add_noise(ones, plan, NoiseDraw(snr_db=draw.snr_db, clip=None, start=None, seed=seed + 1))
    y = y.cpu()
    for u, (o, n) in enumerate(zip(plan.offsets, lens)):
        nu = gauss_noise(seed, u, n)
        a64 = math.sqrt(n / float((nu ** 2).sum()) * 1e4)
        want = a64 * nu
        err = np.abs((y[o:o + n].double().numpy() - 1.0) - want).max() / np.abs(want).max()
        assert err <= 1e-5, (u, err)
    seg = slice(plan.offsets[0], plan.offsets[0] + lens[0])
    assert not torch.equal(other.cpu()[seg], y[seg])


@gpu
def test_clean_cases_and_normalize(fe):
    """snr = +inf, a silent utterance and a zero-energy noise window leave y == x bit for bit; normalize=True is
    wave_stages(normalize=True) of the normalize=False output, bit for bit, and the oracle's normalize_wav of it."""
    g = torch.Generator().manual_seed(8)
    lens = [8000, 6000, 5000, 12000]
    xs = [torch.randn(n, generator=g) for n in lens]
    xs[1] = torch.zeros(lens[1])
    xs[1][::7] = -0.0
    quiet = torch.cat([torch.zeros(6000), torch.randn(100, generator=g)])       # energy only past sample 6000
    bank = lid.NoiseBank([torch.randn(3000, generator=g), quiet])
    plan = fe.make_plan(lens, padded=False)
    packed = fe.pack([x.cuda() for x in xs], plan)
    draw = NoiseDraw(snr_db=torch.tensor([math.inf, 5.0, 5.0, 12.0]), clip=torch.tensor([0, 0, 1, 0]),
                     start=torch.tensor([0, 17, 0, 2999]), seed=0)
    y = fe.add_noise(packed, plan, draw, bank=bank)
    for i in range(3):
        o, n = plan.offsets[i], lens[i]
        assert torch.equal(_bits(y[o:o + n]), _bits(packed[o:o + n])), i
    o, n = plan.offsets[3], lens[3]
    assert not torch.equal(y[o:o + n], packed[o:o + n])
    for gd in (None, 99):                                  # both sources
        b = bank if gd is None else None
        dr = draw if gd is None else NoiseDraw(snr_db=draw.snr_db, clip=None, start=None, seed=gd)
        plain = fe.add_noise(packed, plan, dr, bank=b)
        yn = fe.add_noise(packed, plan, dr, bank=b, normalize=True)
        two = fe.wave_stages(plain, plan, normalize=True)
        assert torch.equal(_bits(yn), _bits(two))
        for i in (0, 2, 3):
            o, n = plan.offsets[i], lens[i]
            want = O.normalize_wav(plain[o:o + n].cpu().unsqueeze(0))[0]
            assert float((yn[o:o + n].cpu() - want).abs().max()) <= 2e-6


@gpu
def test_bad_table_entry_is_nan_not_a_read(fe):
    """An entry the Python layer would reject, passed straight to the ABI: its utterance is NaN, the others are mixed."""
    lens = [4000, 4000]
    plan = fe.make_plan(lens, padded=False)
    bank = lid.NoiseBank([torch.randn(1000), torch.randn(500)])
    x = torch.randn(plan.total_samples, device="cuda")
    tab = torch.tensor([[0, 1000], [1000, 600], [0, 0]], dtype=torch.int64, device="cuda")   # clip 2 runs past the bank
    snr = torch.tensor([10.0, 10.0], device="cuda")
    out = torch.zeros_like(x)
    lib = lid.load_library()
    torch.cuda.synchronize()
    lid._lib.check(lib.lidfe_add_noise(fe.handle, plan.handle, x.data_ptr(), 0, 1.0, out.data_ptr(), bank.data.data_ptr(),
                                       bank.data.numel(), tab.data_ptr(), snr.data_ptr(), 0, 0,
                                       torch.cuda.current_stream().cuda_stream))
    assert bool(torch.isfinite(out[:4000]).all()) and bool(torch.isnan(out[4000:8000]).all())
    with pytest.raises(lid.LidfeError):
        lid._lib.check(lib.lidfe_add_noise(fe.handle, plan.handle, x.data_ptr(), 0, 1.0, x.data_ptr(), None, 0, None,
                                           snr.data_ptr(), 0, 0, None))           # in place
    with pytest.raises(lid.LidfeError):
        lid._lib.check(lib.lidfe_add_noise(fe.handle, plan.handle, x.data_ptr(), 0, 1.0, out.data_ptr(),
                                           bank.data.data_ptr(), bank.data.numel(), None, snr.data_ptr(), 0, 0, None))


def _mixture64(xs, bank, draw):
    """fp64 mixtures (torchaudio.functional.add_noise) rounded to fp32, from the bank draw"""
    out = []
    for i, x in enumerate(xs):
        c = int(draw.clip[i])
        clip = bank.data[bank.offsets[c]:bank.offsets[c] + bank.lengths[c]].cpu()
        y64, _ = _add_noise64(x, _window(clip, int(draw.start[i]), x.numel()), float(draw.snr_db[i]))
        out.append(y64.to(torch.float32))
    return out


@gpu
@pytest.mark.parametrize("kind", ["kaldi", "melspec_db"])
def test_featurize_with_noise(kind):
    f = lid.FrontEnd(n_mels=80, kind=kind)
    g = torch.Generator().manual_seed(31)
    lens = [16000, 7200, 24000, 9000]
    wavs = [O.synth_speechlike(n, 60 + i) for i, n in enumerate(lens)]
    bank = lid.NoiseBank([torch.randn(n, generator=g) for n in (10000, 3000, 32000)])
    aug = lid.NoiseAugment(bank, (0.0, 20.0), generator=torch.Generator().manual_seed(5))
    got, _ = f.featurize(wavs, noise=aug)
    draw = lid.draw_noise(len(lens), (0.0, 20.0), 1.0, bank, torch.Generator().manual_seed(5))
    plan = f.make_plan(lens)
    want = f.featurize_packed(f.add_noise(f.pack(wavs, plan), plan, draw, bank=bank), plan)
    assert torch.equal(got, want)
    if kind == "kaldi":
        got = got.cpu()
        for i, y in enumerate(_mixture64([w[0] for w in wavs], bank, draw)):
            ref = O.kaldi_fbank(y.unsqueeze(0))
            err = float((got[i, :ref.shape[0]] - ref).abs().max() / ref.abs().max())
            assert err <= 3e-4, (i, err)
    # an SNR sweep on one plan: every point equals a fresh call
    packed = f.pack(wavs, plan)
    for snr in (-5.0, 0.0, 10.0, 30.0):
        d = lid.draw_noise(len(lens), snr, 1.0, bank, torch.Generator().manual_seed(9))
        swept = f.featurize_packed(f.add_noise(packed, plan, d, bank=bank), plan)
        fresh_plan = f.make_plan(lens)
        fresh = f.featurize_packed(f.add_noise(f.pack(wavs, fresh_plan), fresh_plan, d, bank=bank), fresh_plan)
        assert torch.equal(swept, fresh), snr
    i16 = lid.FrontEnd(n_mels=80, in_dtype=torch.int16, in_scale=1.0 / 32768)
    with pytest.raises(ValueError):
        i16.featurize([(w[0] * 3000).to(torch.int16) for w in wavs], noise=aug)


def _batch(lens, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(1, n, generator=g) * 0.1, torch.tensor([1, 2, 3]), "utt%d.wav" % i, "en" if i % 2 else "zh")
            for i, n in enumerate(lens)]


@gpu
def test_device_collate_with_noise(fe):
    lens = [16000, 5000, 31000, 12345, 8000]
    batch = _batch(lens, 4)
    l2i = {"en": 0, "zh": 1}
    bank = lid.NoiseBank([torch.randn(n, generator=torch.Generator().manual_seed(n)) for n in (20000, 7000)])
    plain = lid.DeviceCollate(fe, l2i, train=True, mask_times=2)
    noisy = lid.DeviceCollate(fe, l2i, train=True, mask_times=2,
                              noise=lid.NoiseAugment(bank, (0.0, 15.0), generator=torch.Generator().manual_seed(1)))
    torch.manual_seed(123)
    a = plain(batch)[0]
    torch.manual_seed(123)
    b = noisy(batch)[0]
    assert not torch.equal(a, b)
    assert torch.equal(a == 0, b == 0)                    # masks (and padding) exactly where the clean run has them
    clean = lid.DeviceCollate(fe, l2i, train=True, mask_times=2,
                              noise=lid.NoiseAugment(bank, (0.0, 15.0), p=0.0))
    torch.manual_seed(123)
    assert torch.equal(_bits(clean(batch)[0]), _bits(a))
    ev_plain = lid.DeviceCollate(fe, l2i, train=False)(batch)[0]
    ev_noise = lid.DeviceCollate(fe, l2i, train=False, noise=lid.NoiseAugment(None, 0.0))(batch)[0]
    assert torch.equal(_bits(ev_plain), _bits(ev_noise))
    with pytest.raises(ValueError):
        lid.DeviceCollate(lid.FrontEnd(in_dtype=torch.int16, in_scale=1.0 / 32768), l2i, train=True,
                          noise=lid.NoiseAugment(None, 0.0))


@gpu
def test_add_noise_on_a_side_stream(fe):
    """Plan, pack, add_noise and featurize_packed all on a non-current stream, no synchronisation in between: the
    same bits as on the current stream."""
    g = torch.Generator().manual_seed(77)
    lens = [48000, 7000, 128000, 16000]
    wavs = [torch.randn(n, generator=g) for n in lens]
    bank = lid.NoiseBank([torch.randn(50000, generator=g)])
    draw = lid.draw_noise(len(lens), (0.0, 10.0), 1.0, bank, torch.Generator().manual_seed(2))
    plan = fe.make_plan(lens)
    want = fe.featurize_packed(fe.add_noise(fe.pack(wavs, plan), plan, draw, bank=bank, normalize=True), plan).cpu()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side_plan = fe.make_plan(lens, stream=s)
        packed = fe.pack(wavs, side_plan)
        mixed = fe.add_noise(packed, side_plan, draw, bank=bank, normalize=True, stream=s)
        feats = torch.empty((len(lens), side_plan.t_max, 80), device="cuda")
        fe.featurize_packed(mixed, side_plan, out=feats, stream=s)
    torch.cuda.current_stream().wait_stream(s)
    assert torch.equal(feats.cpu(), want)
