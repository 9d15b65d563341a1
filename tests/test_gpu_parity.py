"""GPU parity: the sm_100a path (through the C ABI, via speech_lid_b200) against the oracle and the committed
reference fixtures.  Run on the B200 box: python -m pytest tests -m gpu.

Acceptance metrics (SURVEY.md §8c).  Elementwise rtol=1e-4 is not met by the reference against an fp64 evaluation
of itself: with preemph=1.0 the three lowest mel bins of white noise are cancellation dominated, the fp32 FFT round-off
(~eps * |X_nyquist|) is amplified by the log wherever such a bin happens to be nearly empty, and the reference's OWN
fp32 error there reaches ~9e-4 abs (8e-5 of the feature range) on a handful of 8-s utterances.  Two independent fp32
pipelines therefore cannot agree to 1e-4 of the range in those bins on every utterance; the metrics are:
  (i)   frame counts, mask bounds and masked positions: integer / bit exact;
  (ii)  per utterance  max|gpu - oracle32| / max|oracle32|  <= 1e-4 over mel bins >= 3 (77 of 80 dims), over ALL bins
        for speech-like input and for MFCC;  <= 3e-4 over bins 0-2 of white noise (cancellation dominated);
  (iii) at most 0.01 % of the elements violate isclose(rtol=1e-4, atol=5e-4);
  (iv)  "no worse than the reference": per mel-bin group (0-2, 3-9, >=10), the median and the 99th percentile of
        |gpu - truth64| are <= 1.5 x those of |oracle32 - truth64|, and max|gpu - truth64| <= 4 x max|oracle32 - truth64|
        (heavy-tailed errors: rms and max over ~800 frames are too noisy for a tighter bound);
  (v)   speech-like input (low bins carry energy): norm-relative <= 1e-4 on all bins and isclose(rtol=1e-4, atol=1e-5)
        on >= 99.9 % of elements.
"""
import os

import numpy as np
import pytest
import torch

from oracle import frontend_oracle as O

pytestmark = pytest.mark.gpu

NORM_REL = 1e-4


@pytest.fixture(scope="module")
def lid():
    import speech_lid_b200 as m
    return m


@pytest.fixture(scope="module")
def fe(lid):
    return lid.FrontEnd(n_mels=80)


def _norm_rel(got, want):
    return float((got - want).abs().max() / want.abs().max())


def _cuda_kernels(fn):
    """Names of the CUDA kernels that fn() launches (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


LOW_BINS = 3            # mel bins 0..2: cancellation dominated for white noise through the 1.0 pre-emphasis
NORM_REL_LOW = 3e-4
DEEP_NULL = 9.2         # nepers (40 dB) below the mel bin's median energy over the utterance
DEEP_NULL_ENERGY = 1e-6  # allowed |E_gpu - E_ref| there, in units of that median energy (about 8 fp32 ulps of it)


def _deep_nulls(want):
    """Deep spectral nulls: frames whose energy in a mel bin lies more than 40 dB under that bin's median.  The FFT
    round-off of ANY fp32 pipeline is relative to the typical magnitude in the frame, not to the nearly empty bin, so
    the log amplifies it without bound there (one such point per ~1e5 in white noise; the fp32 reference itself is off
    by 3e-4 .. 1e-3 against fp64 on them, and WHICH way depends on the host CPU's FFT kernels).  They are checked in
    the energy domain against the fp32 resolution of the bin's typical energy instead."""
    live = want != 0.0                                     # SpecAugment zeros are compared exactly elsewhere
    med = torch.where(live, want, torch.full_like(want, float("nan"))).nanmedian(0).values
    med = torch.nan_to_num(med, nan=0.0)
    return live & (want < med - DEEP_NULL), med


def _check_fbank(got, want, what, all_bins=False):
    """Metric (ii) + (iii).  got/want: (T, 80) log-mel."""
    assert got.shape == want.shape, what
    assert torch.isfinite(got).all(), what
    scale = want.abs().max()
    deep, med = _deep_nulls(want)
    err = (got - want).abs().masked_fill(deep, 0.0)
    hi = float(err[:, LOW_BINS:].max() / scale)
    lo = float(err[:, :LOW_BINS].max() / scale)
    assert hi <= NORM_REL, "%s: norm-relative error %g on bins >= %d" % (what, hi, LOW_BINS)
    assert lo <= (NORM_REL if all_bins else NORM_REL_LOW), "%s: norm-relative error %g on bins < %d" % (what, lo, LOW_BINS)
    if deep.any():
        assert deep.float().mean().item() <= 1e-3, "%s: %d deep nulls?" % (what, int(deep.sum()))
        e = ((got.double().exp() - want.double().exp()).abs() / med.double().exp())[deep].max().item()
        assert e <= DEEP_NULL_ENERGY, "%s: energy error %g (x median bin energy) in a deep null" % (what, e)
    bad = 1.0 - torch.isclose(got, want, rtol=1e-4, atol=5e-4).float().mean().item()
    assert bad <= 1e-4, "%s: %.4f %% of elements outside rtol=1e-4, atol=5e-4" % (what, 100 * bad)


def test_extension_is_loaded(lid):
    lib = lid.load_library()
    assert lib.lidfe_abi_version() == lid._lib.ABI_VERSION
    with open("/proc/self/maps") as f:
        assert "liblidfe.so" in f.read()


def test_fbank_vs_reference_fixtures(fe, golden_dir):
    z = np.load(os.path.join(golden_dir, "fbank_kaldi.npz"))
    for name in [k[3:] for k in z.files if k.startswith("in_")]:
        x = torch.from_numpy(z["in_" + name])
        want = torch.from_numpy(z["out_" + name])[0].T.contiguous()        # (T, 80)
        feats, percents = fe.featurize([x])
        got = feats[0].cpu()
        assert got.shape[0] == O.kaldi_num_frames(x.shape[-1]) == want.shape[0]
        assert percents.tolist() == [1.0]
        if name == "silence":
            assert torch.equal(got, want)                                   # exactly log(eps) everywhere
        else:
            _check_fbank(got, want, name)


def test_cfg1_batch_vs_oracle(fe):
    """BASELINE config 1: 32 x 3 s, 80-dim kaldi fbank."""
    wavs = [O.synth_noise(48000, 100 + i) for i in range(32)]
    feats, percents = fe.featurize(wavs)
    assert feats.shape == (32, 298, 80) and torch.all(percents == 1.0)
    feats = feats.cpu()
    worst = 0.0
    for i, w in enumerate(wavs):
        want = O.kaldi_fbank(w)
        _check_fbank(feats[i], want, "utt %d" % i)
        worst = max(worst, _norm_rel(feats[i], want))
    print("cfg1 worst norm-relative error %.3g" % worst)


def test_no_worse_than_reference_vs_fp64(fe):
    """Metric (iv): both fp32 pipelines against an fp64 evaluation with the same fp32 tables.  The error of a
    cancellation-dominated low bin is heavy tailed (the log amplifies the FFT round-off wherever the bin is nearly
    empty), so the distributions are compared at their median and 99th percentile, pooled over 4 utterances, plus
    a loose bound on the maximum outside the deep nulls (see _deep_nulls), which are bounded in the energy domain."""
    groups = ((0, 3), (3, 10), (10, 80))
    ref_e, gpu_e = [], []
    for seed in range(4):
        x = O.synth_noise(128000, 200 + seed)
        got = fe.featurize([x])[0][0].cpu().double()
        truth = O.truth64_fbank(x)
        deep, med = _deep_nulls(truth.float())
        if deep.any():
            e = ((got.exp() - truth.exp()).abs() / med.double().exp())[deep].max().item()
            assert e <= DEEP_NULL_ENERGY, "energy error %g (x median bin energy) in a deep null" % e
        ref_e.append((O.kaldi_fbank(x).double() - truth).abs().masked_fill(deep, 0.0))
        gpu_e.append((got - truth).abs().masked_fill(deep, 0.0))
    ref_e, gpu_e = torch.cat(ref_e), torch.cat(gpu_e)
    for a, b in groups:
        r, g = ref_e[:, a:b].flatten(), gpu_e[:, a:b].flatten()
        for q in (0.5, 0.99):
            rq, gq = torch.quantile(r, q).item(), torch.quantile(g, q).item()
            assert gq <= 1.5 * rq + 2e-7, "bins [%d,%d) q%.2f: gpu %g vs reference %g" % (a, b, q, gq, rq)
        assert g.max().item() <= 4.0 * r.max().item() + 2e-5, "bins [%d,%d): max gpu %g vs reference %g" % (
            a, b, g.max().item(), r.max().item())


def test_speechlike_plain_rtol(fe):
    for seed in range(3):
        x = O.synth_speechlike(64000, 300 + seed)
        got = fe.featurize([x])[0][0].cpu()
        want = O.kaldi_fbank(x)
        _check_fbank(got, want, "speech %d" % seed, all_bins=True)
        ok = torch.isclose(got, want, rtol=1e-4, atol=1e-5).float().mean().item()
        assert ok >= 0.999, "only %.5f of elements within rtol=1e-4" % ok


def test_ragged_batch_padded_and_packed(fe):
    """Variable lengths: padded (B, T_max, 80) with zero rows + wav_percents, and the packed layout."""
    lens = [400, 559, 560, 16000, 5000, 12345, 31999, 720, 8000, 16001]
    wavs = [O.synth_noise(n, 400 + i) for i, n in enumerate(lens)]
    want = [O.kaldi_fbank(w) for w in wavs]
    ref_batch, ref_percents = O.collate_features([w.T.unsqueeze(0) for w in want])
    feats, percents = fe.featurize(wavs, padded=True)
    feats = feats.cpu()
    assert feats.shape == ref_batch.shape
    assert torch.equal(percents, ref_percents)
    for i, w in enumerate(want):
        T = w.shape[0]
        _check_fbank(feats[i, :T], w, "ragged %d" % i)
        assert torch.all(feats[i, T:] == 0.0), "padding rows of utt %d are not zero" % i
    packed, _ = fe.featurize(wavs, padded=False)
    assert packed.shape == (sum(w.shape[0] for w in want), 80)
    assert torch.equal(packed.cpu(), torch.cat([feats[i, :w.shape[0]] for i, w in enumerate(want)]))


def test_unaligned_offsets_fallback(fe):
    """Utterances packed back to back at odd offsets take the element-load staging path: same numbers."""
    lens = [1001, 4003, 777]
    wavs = [O.synth_noise(n, 500 + i) for i, n in enumerate(lens)]
    offs = [1, 1 + 1001 + 2, 1 + 1001 + 2 + 4003 + 1]
    buf = torch.zeros(offs[-1] + lens[-1] + 3)
    for w, o in zip(wavs, offs):
        buf[o:o + w.shape[-1]] = w[0]
    plan = fe.make_plan(lens, padded=False, offsets=offs)
    out = fe.featurize_packed(buf.cuda(), plan).cpu()
    aligned, _ = fe.featurize(wavs, padded=False)
    assert torch.equal(out, aligned.cpu())


def test_short_utterance_raises(fe):
    with pytest.raises(AssertionError):
        fe.featurize([torch.zeros(1, 399)])


def test_mfcc_vs_fixtures_and_oracle(lid, golden_dir):
    mf = lid.FrontEnd(n_mels=80, n_ceps=40)
    z = np.load(os.path.join(golden_dir, "mfcc_kaldi.npz"))
    for name in [k[3:] for k in z.files if k.startswith("in_")]:
        x = torch.from_numpy(z["in_" + name])
        want = torch.from_numpy(z["out_" + name])
        got = mf.featurize([x])[0][0].cpu()
        assert got.shape == want.shape
        assert _norm_rel(got, want) <= NORM_REL, name
    wavs = [O.synth_noise(64000, 600 + i) for i in range(4)]      # BASELINE config 3 shape (4 of 512)
    feats, _ = mf.featurize(wavs)
    assert feats.shape == (4, 398, 40)
    for i, w in enumerate(wavs):
        assert _norm_rel(feats[i].cpu(), O.kaldi_mfcc(w)) <= NORM_REL


def test_generic_kernel_variant_configs(lid):
    """Configurations outside the two unrolled kernel variants (Kaldi-80 call, HTK-80 stft call) run the generic
    variant: runtime mel loop, coefficient-c pre-emphasis, in-kernel DCT epilogue when n_mels % 4 != 0 or statistics
    are needed.  Oracle = the same torchaudio arithmetic with those arguments."""
    for n_mels, pre in ((40, 0.97), (64, 1.0), (23, 0.97)):
        fe = lid.FrontEnd(n_mels=n_mels, preemph=pre)
        for kind, gen, all_bins in (("noise", O.synth_noise, False), ("speech", O.synth_speechlike, True)):
            wavs = [gen(n, 900 + i) for i, n in enumerate((32000, 5000, 16000))]
            feats, _ = fe.featurize(wavs)
            feats = feats.cpu()
            for i, w in enumerate(wavs):
                want = O.kaldi_fbank(w, n_mels=n_mels, preemph=pre)
                _check_fbank(feats[i, :want.shape[0]], want, "%s n_mels=%d preemph=%g utt %d" % (kind, n_mels, pre, i),
                             all_bins=all_bins)
                assert torch.all(feats[i, want.shape[0]:] == 0)
    # classic Kaldi MFCC: 13 cepstra of 23 mel bins, 0.97 pre-emphasis (DCT epilogue inside the fbank kernel)
    mf = lid.FrontEnd(n_mels=23, n_ceps=13, preemph=0.97)
    wavs = [O.synth_noise(n, 950 + i) for i, n in enumerate((32000, 7000))]
    feats, _ = mf.featurize(wavs)
    assert feats.shape == (2, 198, 13)
    for i, w in enumerate(wavs):
        want = O.kaldi_mfcc(w, num_ceps=13, n_mels=23, preemph=0.97)
        assert _norm_rel(feats[i, :want.shape[0]].cpu(), want) <= NORM_REL
    # MFCC-40 + per-utterance CMVN: statistics force the in-kernel DCT variant; tight against the device's own raw
    # cepstra, loose against the oracle chain (1/std amplifies the fbank round-off)
    mf = lid.FrontEnd(n_mels=80, n_ceps=40)
    wavs = [O.synth_speechlike(n, 960 + i) for i, n in enumerate((48000, 20000))]
    raw, _ = mf.featurize(wavs)
    norm, _ = mf.featurize(wavs, cmvn="utt")
    for i, w in enumerate(wavs):
        T = O.kaldi_num_frames(w.shape[-1])
        want = O.cmvn_per_utt(raw[i, :T].cpu())
        assert torch.allclose(norm[i, :T].cpu(), want, rtol=1e-4, atol=2e-4), (norm[i, :T].cpu() - want).abs().max()
        full = O.cmvn_per_utt(O.kaldi_mfcc(w))
        assert torch.allclose(norm[i, :T].cpu(), full, rtol=1e-3, atol=5e-3), (norm[i, :T].cpu() - full).abs().max()
    # MFCC of n_mels % 8 == 4 mel bins through the two-kernel path (the tensor-core DCT's last k-step has four mel bins):
    # ragged padded batch, masks, global CMVN with the raw cepstra's own statistics.  Against the oracle chain, and
    # against the device's own log-mels times the DCT and lifter in fp64 (the bound of the cfg3 linearity test).  Both
    # bounds are relative to the range of the raw cepstra, so the normalised output's error is taken back to cepstral
    # units first: global CMVN multiplies column j's error by 1 / std_j, and a high cepstrum's std is far below the range
    from speech_lid_b200 import tables
    for n_mels, n_ceps in ((60, 40), (20, 13)):
        mf, fb = lid.FrontEnd(n_mels=n_mels, n_ceps=n_ceps), lid.FrontEnd(n_mels=n_mels)
        lens = (48000, 7000, 20000)
        wavs = [O.synth_speechlike(n, 970 + i) for i, n in enumerate(lens)]
        frames = [O.kaldi_num_frames(n) for n in lens]
        plan, plan_f = mf.make_plan(lens, padded=True), fb.make_plan(lens, padded=True)
        packed = mf.pack(wavs, plan)
        raw = mf.featurize_packed(packed, plan).cpu()
        stats = O.cmvn_stats([raw[i, :T] for i, T in enumerate(frames)]).cuda()
        torch.manual_seed(13)
        masks = lid.draw_masks(frames, n_ceps, 0.05, n_ceps // 4, 2).cuda()
        got, names = _cuda_kernels(lambda: mf.featurize_packed(packed, plan, masks=masks, cmvn="global_apply",
                                                               stats_in=stats).cpu())
        assert any("mfcc_dct_mma_kernel" in n for n in names), names
        logmel = fb.featurize_packed(fb.pack(wavs, plan_f), plan_f).double()
        lin = ((logmel @ tables.dct_matrix(n_ceps, n_mels).cuda().double()) * tables.lifter(n_ceps, 22.0).cuda().double()).cpu()
        mean, std = O.cmvn_finalize(stats.cpu())
        for i, (w, T) in enumerate(zip(wavs, frames)):
            b = [tuple(int(v) for v in masks[i, q]) for q in range(masks.shape[1])]
            mask = lambda x: O.apply_mask_bounds(x.T.unsqueeze(0), b)[0].T        # noqa: E731
            ceps = O.kaldi_mfcc(w, num_ceps=n_ceps, n_mels=n_mels)
            rel = float((raw[i, :T].double() - lin[i, :T]).abs().max() / lin[i, :T].abs().max())
            assert rel < 2e-6, (n_mels, i, rel)
            assert _norm_rel(raw[i, :T], ceps) <= NORM_REL, (n_mels, i, _norm_rel(raw[i, :T], ceps))
            want64 = mask((lin[i, :T] - mean) / (std + O.CMVN_EPS))
            rel = float(((got[i, :T].double() - want64).abs() * (std + O.CMVN_EPS)).max() / lin[i, :T].abs().max())
            assert rel < 2e-6, (n_mels, i, rel)
            want = mask(O.cmvn_apply(ceps, mean, std)).double()
            rel = float(((got[i, :T].double() - want).abs() * (std + O.CMVN_EPS)).max() / ceps.abs().max())
            assert rel <= NORM_REL, (n_mels, i, rel)
            assert torch.all(got[i, T:] == 0)


def test_specaug_masks_bit_exact(fe, lid, golden_dir):
    """Masks drawn on the host from the reference's RNG stream, applied in the kernel epilogue: the masked
    positions are exactly the reference's, and every unmasked value equals the unmasked run bit for bit."""
    z = np.load(os.path.join(golden_dir, "specaug.npz"))
    spec_ref = torch.from_numpy(z["spec_t798_default"])
    out_ref = torch.from_numpy(z["out_t798_default"])
    t_mask, f_mask, mask_times, seed = z["kw_t798_default"]
    x = O.synth_noise(128000, int(seed))
    torch.manual_seed(int(seed))
    masks = lid.draw_masks([798], 80, float(t_mask), int(f_mask), int(mask_times))
    plain = fe.featurize([x])[0][0].cpu()
    masked = fe.featurize([x], masks=masks)[0][0].cpu()
    zero_ref = (out_ref[0].T == 0.0) & (spec_ref[0].T != 0.0)
    assert torch.equal(masked == 0.0, zero_ref | (plain == 0.0))
    assert torch.equal(masked[~zero_ref], plain[~zero_ref])
    # batch: per-utterance tables in batch order, different lengths
    lens = [128000, 48000, 3300, 16000]
    wavs = [O.synth_noise(n, 700 + i) for i, n in enumerate(lens)]
    frames = [O.kaldi_num_frames(n) for n in lens]
    torch.manual_seed(99)
    masks = lid.draw_masks(frames, 80, 0.05, 27, 2)
    torch.manual_seed(99)
    want = [O.spectrogram_augment(O.wav2mel_kaldi(w), 0.05, 27, 2)[0].T for w in wavs]
    got, _ = fe.featurize(wavs, masks=masks)
    got = got.cpu()
    for i, w in enumerate(want):
        assert torch.equal(got[i, :frames[i]] == 0.0, w == 0.0), "mask positions of utt %d" % i
        _check_fbank(got[i, :frames[i]], w, "masked utt %d" % i)


def test_per_utt_cmvn(fe, lid):
    lens = [128000, 20000, 48000]
    wavs = [O.synth_noise(n, 800 + i) for i, n in enumerate(lens)]
    frames = [O.kaldi_num_frames(n) for n in lens]
    torch.manual_seed(5)
    masks = lid.draw_masks(frames, 80, 0.05, 27, 2)
    got, _ = fe.featurize(wavs, masks=masks, cmvn="utt")
    got = got.cpu()
    raw, _ = fe.featurize(wavs)
    raw = raw.cpu()
    for i in range(len(lens)):
        T = frames[i]
        # our CMVN definition applied to the device's own raw features: isolates the normalisation arithmetic
        want = O.cmvn_per_utt(raw[i, :T])
        b = [tuple(int(v) for v in masks[i, q]) for q in range(masks.shape[1])]
        want = O.apply_mask_bounds(want.T.unsqueeze(0), b)[0].T
        assert torch.allclose(got[i, :T], want, rtol=1e-5, atol=2e-6), (got[i, :T] - want).abs().max()
        # and end to end against the oracle chain
        full = O.apply_mask_bounds(O.cmvn_per_utt(O.kaldi_fbank(wavs[i])).T.unsqueeze(0), b)[0].T
        assert torch.allclose(got[i, :T], full, rtol=1e-3, atol=2e-3)
        assert torch.all(got[i, T:] == 0)


def test_repeated_launches_streams_and_mask_limits(fe, lid):
    """The per-utterance statistics workspace is double buffered and cleared by the apply kernel of the previous
    launch: repeated launches on one plan, launches on side streams, and the maximum number of masks must all give the
    same bits as a first launch."""
    lens = [48000, 7000, 128000, 16000, 400]
    wavs = [O.synth_noise(n, 1000 + i).squeeze(0) for i, n in enumerate(lens)]
    frames = [O.kaldi_num_frames(n) for n in lens]
    plan = fe.make_plan(lens, padded=True)
    packed = fe.pack([w.cuda() for w in wavs], plan)
    torch.manual_seed(11)
    masks = lid.draw_masks(frames, 80, 0.05, 27, 8).cuda()                 # 8 (time, freq) mask rows: the ABI maximum
    assert masks.shape[1] == 8
    same = lambda x, y: torch.equal(torch.nan_to_num(x, nan=-777.0), torch.nan_to_num(y, nan=-777.0))   # noqa: E731
    first = fe.featurize_packed(packed, plan, masks=masks, cmvn="utt").clone()
    assert torch.isnan(first[4, 0]).any()      # one frame: the unbiased std of one sample is NaN, as torch.std gives
    for _ in range(5):                                                     # ping-pong halves, both parities
        again = fe.featurize_packed(packed, plan, masks=masks, cmvn="utt")
        assert same(again, first)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    plan2 = fe.make_plan(lens, padded=True)
    torch.cuda.synchronize()
    a = fe.featurize_packed(packed, plan, masks=masks, cmvn="utt", stream=s1)
    b = fe.featurize_packed(packed, plan2, masks=masks, cmvn="utt", stream=s2)    # same handle, other plan, concurrently
    c = fe.featurize_packed(packed, plan, cmvn="none", stream=s1)
    torch.cuda.synchronize()
    assert same(a, first) and same(b, first)
    raw = fe.featurize_packed(packed, plan, cmvn="none")
    assert torch.equal(c, raw)
    # masks land where the table says
    for i, T in enumerate(frames[:-1]):
        for q in range(8):
            t0, t1, f0, f1 = (int(v) for v in masks[i, q])
            assert torch.all(first[i, t0:t1] == 0) and torch.all(first[i, :T, f0:f1] == 0)
        assert torch.isfinite(first[i, :T]).all()
    with pytest.raises(Exception):
        fe.featurize_packed(packed, plan, masks=torch.zeros(len(lens), 9, 4, dtype=torch.int32).cuda())   # > 8 masks


def test_global_cmvn_two_pass(fe):
    lens = [30000, 16000, 64000, 8000]
    wavs = [O.synth_noise(n, 900 + i) for i, n in enumerate(lens)]
    plan = fe.make_plan(lens, padded=False)
    packed = fe.pack(wavs, plan)
    stats = torch.zeros(161, dtype=torch.float64, device="cuda")
    raw = fe.featurize_packed(packed, plan, cmvn="global_accum", stats_out=stats)
    rows = raw.cpu()
    want_stats = O.cmvn_stats([rows])
    assert stats[160].item() == rows.shape[0]
    assert torch.allclose(stats.cpu(), want_stats, rtol=1e-6, atol=1e-4)
    mean, std = O.cmvn_finalize(stats.cpu())
    want = O.cmvn_apply(rows, mean, std)
    two_pass = fe.cmvn_apply(raw.clone(), plan, stats).cpu()
    assert torch.allclose(two_pass, want, rtol=1e-5, atol=2e-6)
    fused = fe.featurize_packed(packed, plan, cmvn="global_apply", stats_in=stats).cpu()
    assert torch.allclose(fused, want, rtol=1e-5, atol=2e-6)


def test_int16_input(lid):
    fe16 = lid.FrontEnd(n_mels=80, in_dtype=torch.int16, in_scale=1.0 / 32768.0)
    g = torch.Generator().manual_seed(3)
    pcm = (torch.randn(1, 40000, generator=g) * 3000).clamp(-32768, 32767).to(torch.int16)
    got = fe16.featurize([pcm])[0][0].cpu()
    want = O.kaldi_fbank(pcm.float() * (1.0 / 32768.0))
    _check_fbank(got, want, "int16")


def test_wave_stages(fe, golden_dir):
    z = np.load(os.path.join(golden_dir, "waveform_stages.npz"))
    raw = torch.from_numpy(z["raw"])
    plan = fe.make_plan([raw.shape[-1]], padded=False)
    packed = fe.pack([raw], plan)
    norm = fe.wave_stages(packed, plan, normalize=True).cpu()[:raw.shape[-1]]
    assert torch.allclose(norm, torch.from_numpy(z["normalized"])[0], rtol=2e-6, atol=2e-6)
    noise = fe.pack([torch.from_numpy(z["dither_noise"])], plan)
    dith = fe.wave_stages(packed, plan, dither=1e-5, noise=noise)
    aug = fe.wave_stages(dith, plan, preemph=0.97).cpu()[:raw.shape[-1]]
    assert torch.equal(aug, torch.from_numpy(z["augmented"])[0])       # same fp32 op order -> bit exact


def test_dropin_audio_processor(lid, golden_dir):
    from speech_lid_b200 import audio_processor as ap
    z = np.load(os.path.join(golden_dir, "fbank_kaldi.npz"))
    x = torch.from_numpy(z["in_noise_1s"])
    want = torch.from_numpy(z["out_noise_1s"])
    got = ap.wav2mel(x, use_kaildi=True)
    assert got.shape == want.shape == (1, 80, 98) and got.device.type == "cpu"
    _check_fbank(got[0].T, want[0].T, "drop-in wav2mel")
    assert ap.wav2mel(x.cuda(), use_kaildi=True).is_cuda
    with pytest.raises(AssertionError):
        ap.wav2mel(torch.zeros(1, 100), use_kaildi=True)
    torch.manual_seed(11)
    a = ap.spectrogram_augment(want, mask_times=2)
    torch.manual_seed(11)
    b = O.spectrogram_augment(want, mask_times=2)
    assert torch.equal(a, b)
    assert ap.spectrogram_augment(want, mask_times=0) is want
    # stereo input: dither + pre-emphasis are element-wise per channel; normalize_wav only broadcasts for mono, in the
    # reference as here (ref: lid/audio_processor.py:112-113, 128-134)
    st = torch.stack([x[0], 0.3 * x[0].flip(0) + 0.01], 0)
    with pytest.raises(RuntimeError):
        O.normalize_wav(st)
    with pytest.raises(RuntimeError):
        ap.normalize_wav(st)
    torch.manual_seed(5)
    a2, _ = ap.wav_augment(st.clone(), 16000)
    torch.manual_seed(5)
    w2 = st.clone()
    w2 += 1e-5 * torch.rand_like(w2)
    b2 = torch.cat((w2[:, 0].unsqueeze(1), w2[:, 1:] - 0.97 * w2[:, :-1]), dim=1)
    assert torch.equal(a2, b2)


def test_full_size_properties(fe, lid):
    """BASELINE config 2 at full size (256 x 8 s): properties that do not need the CPU oracle at that size."""
    g = torch.Generator(device="cuda").manual_seed(1)
    wav = torch.randn(256, 128000, device="cuda", generator=g)
    plan = fe.make_plan([128000] * 256, padded=True)
    out = fe.featurize_packed(wav.reshape(-1), plan)
    assert out.shape == (256, 798, 80) and torch.isfinite(out).all()
    # determinism / idempotence
    assert torch.equal(out, fe.featurize_packed(wav.reshape(-1), plan))
    # shift property: utterance i delayed by one hop reproduces frames 1.. of the original bit for bit
    shifted = torch.randn(256, 128000, device="cuda")
    shifted[:, :-160] = wav[:, 160:]
    out2 = fe.featurize_packed(shifted.reshape(-1), plan)
    assert torch.equal(out2[:, :-1], out[:, 1:])
    # spot-check 3 utterances against the oracle
    for i in (0, 101, 255):
        _check_fbank(out[i].cpu(), O.kaldi_fbank(wav[i].cpu()), "full-size utt %d" % i)
    # per-utterance CMVN at full size: zero mean / unit (unbiased) std per utterance and bin
    y = fe.featurize_packed(wav.reshape(-1), plan, cmvn="utt")
    assert y.mean(1).abs().max() < 1e-4 and (y.std(1) - 1).abs().max() < 1e-4


def test_melspec_db_default_branch(lid, golden_dir):
    """Row A9 -- the reference's DEFAULT wav2mel branch: MelSpectrogram + AmplitudeToDB(top_db=80), pad 0 / 16, against
    outputs of the reference itself (tests/golden/melspec_db.npz) and the oracle on a ragged batch."""
    from speech_lid_b200 import audio_processor as ap
    z = np.load(os.path.join(golden_dir, "melspec_db.npz"))
    fes = {}
    for name in [k[3:] for k in z.files if k.startswith("in_")]:
        x = torch.from_numpy(z["in_" + name])
        pad = int(z["pad_" + name][0])
        want = torch.from_numpy(z["out_" + name])                       # (1, 80, T)
        fe = fes.setdefault(pad, lid.FrontEnd(kind="melspec_db", pad=pad))
        feats, percents = fe.featurize([x])
        got = feats[0].cpu()
        assert got.shape == (want.shape[2], 80) and want.shape[2] == O.num_frames_centered(x.shape[-1], pad=pad)
        assert _norm_rel(got, want[0].T) <= NORM_REL, "%s: %g" % (name, _norm_rel(got, want[0].T))
        assert torch.allclose(got, want[0].T, rtol=1e-4, atol=2e-4), (name, float((got - want[0].T).abs().max()))
        # the top_db clamp floor is the utterance max - 80
        assert abs(float(got.min()) - max(float(want.min()), float(want.max()) - 80.0)) < 1e-3
        # drop-in call, default branch
        got2 = ap.wav2mel(x, pad=pad)
        assert got2.shape == want.shape and _norm_rel(got2, want) <= NORM_REL
    # ragged batch incl. utterances shorter than one tile and edge-only utterances (every tile reflects)
    lens = [16000, 300, 2560, 40000, 257, 12345]
    wavs = [O.synth_noise(n, 950 + i) for i, n in enumerate(lens)]
    wavs[3] = torch.cat([wavs[3][:, :20000], 1e-5 * wavs[3][:, 20000:]], 1)       # makes the clamp bite
    fe = fes[0]
    feats, percents = fe.featurize(wavs)
    feats = feats.cpu()
    for i, w in enumerate(wavs):
        want = O.melspec_db(w)[0].T
        T = want.shape[0]
        assert _norm_rel(feats[i, :T], want) <= NORM_REL, i
        assert torch.all(feats[i, T:] == 0)
    assert abs(float(feats[3, :O.num_frames_centered(40000)].min()) - (float(O.melspec_db(wavs[3]).max()) - 80.0)) < 1e-3
    # SpecAugment on top (masks after the clamp, as the reference composes them)
    frames = [O.num_frames_centered(n) for n in lens]
    torch.manual_seed(3)
    masks = lid.draw_masks(frames, 80, 0.05, 27, 2)
    torch.manual_seed(3)
    ref = [O.spectrogram_augment(O.melspec_db(w), 0.05, 27, 2)[0].T for w in wavs]
    got, _ = fe.featurize(wavs, masks=masks)
    for i, r in enumerate(ref):
        g = got[i, :frames[i]].cpu()
        assert torch.equal(g == 0, r == 0) and _norm_rel(g, r) <= NORM_REL
    with pytest.raises(RuntimeError):
        ap.wav2mel(torch.zeros(1, 200))                                            # reflect padding >= input length


def test_cfg3_mfcc_full_size_properties(lid):
    """BASELINE config 3 at full size (512 x 4 s, 40 MFCC of 80 mel): shape, determinism, spot checks, linearity of
    the DCT epilogue (MFCC == log-mel @ DCT * lifter computed from the fbank path's own output)."""
    from speech_lid_b200 import tables
    mf = lid.FrontEnd(n_mels=80, n_ceps=40)
    fb = lid.FrontEnd(n_mels=80)
    g = torch.Generator(device="cuda").manual_seed(2)
    wav = torch.randn(512, 64000, device="cuda", generator=g)
    plan_m = mf.make_plan([64000] * 512, padded=True)
    plan_f = fb.make_plan([64000] * 512, padded=True)
    c = mf.featurize_packed(wav.reshape(-1), plan_m)
    assert c.shape == (512, 398, 40) and torch.isfinite(c).all()
    assert torch.equal(c, mf.featurize_packed(wav.reshape(-1), plan_m))
    logmel = fb.featurize_packed(wav.reshape(-1), plan_f)
    dct = tables.dct_matrix(40, 80).cuda().double()
    lift = tables.lifter(40, 22.0).cuda().double()
    want = (logmel.double() @ dct) * lift
    assert float((c.double() - want).abs().max() / want.abs().max()) < 2e-6
    for i in (0, 255, 511):
        assert _norm_rel(c[i].cpu(), O.kaldi_mfcc(wav[i].cpu())) <= NORM_REL


def test_host_buffer_entry_matches_device_entry(fe, lid):
    """featurize_host (pinned host in / out, 8 pipelined utterance groups) == featurize_packed on the same data."""
    lens = [20000 + 977 * i for i in range(37)]
    wavs = [O.synth_noise(n, 1200 + i) for i, n in enumerate(lens)]
    plan = fe.make_plan(lens, padded=True)
    host_in = torch.zeros(plan.total_samples).pin_memory()
    for w, o, n in zip(wavs, plan.offsets, lens):
        host_in[o:o + n] = w[0]
    torch.manual_seed(8)
    masks = lid.draw_masks(plan.frames, 80, 0.05, 27, 2)
    host_out = torch.empty(len(lens), plan.t_max, 80).pin_memory()
    fe.featurize_host(host_in, plan, host_out, masks=masks, cmvn="utt")
    dev = fe.featurize_packed(host_in.cuda(), plan, masks=masks, cmvn="utt").cpu()
    assert torch.allclose(host_out, dev, rtol=0, atol=2e-6)      # per-utterance sums are added in a different order
    assert torch.equal(host_out == 0, dev == 0)


def test_int16_pcm_host_pipeline(fe, lid):
    """Row f2: host ships raw int16 PCM; scaling by 1/32768 + normalize_wav run on the device before framing."""
    g = torch.Generator().manual_seed(11)
    lens = [16000, 23456, 9000, 40000, 12000]
    pcm = [(torch.randn(1, n, generator=g) * 2500 + 30).clamp(-32768, 32767).to(torch.int16) for n in lens]
    plan = fe.make_plan(lens, padded=True)
    host_in = torch.zeros(plan.total_samples, dtype=torch.int16).pin_memory()
    for w, o, n in zip(pcm, plan.offsets, lens):
        host_in[o:o + n] = w[0]
    host_out = torch.empty(len(lens), plan.t_max, 80).pin_memory()
    fe.featurize_host(host_in, plan, host_out, chunks=2)
    for i, w in enumerate(pcm):
        want = O.kaldi_fbank(O.normalize_wav(w.float() * (1.0 / 32768.0)))
        _check_fbank(host_out[i, :want.shape[0]], want, "pcm utt %d" % i)


def test_device_collate_matches_reference_collate(lid, golden_dir):
    """DeviceCollate on ``type: wav`` items == the reference's collate on ``type: mel`` items
    (ref: lid/raw_datasets.py:345-365; golden collate.npz was produced by the reference's wav2mel + pad_sequence)."""
    z = np.load(os.path.join(golden_dir, "collate.npz"))
    lang2index = {"Persian": 0, "Swahili": 1, "Vietnamese": 2}
    g = torch.Generator().manual_seed(8)
    batch = []
    for i, lang in enumerate(("Vietnamese", "Persian", "Swahili")):
        batch.append((torch.from_numpy(z["in_%d" % i]), torch.randint(1, 30, (5 + 3 * i,), generator=g), "f%d.wav" % i, lang))
    fe = lid.FrontEnd(n_mels=80)
    wavs, texts, wav_percents, text_percents, paths, langs = lid.DeviceCollate(fe, lang2index)(batch)
    want = torch.from_numpy(z["wavs"])
    assert wavs.is_cuda and wavs.shape == want.shape
    for i in range(3):
        T = O.kaldi_num_frames(batch[i][0].shape[-1])
        _check_fbank(wavs[i, :T].cpu(), want[i, :T], "collate utt %d" % i)
        assert torch.all(wavs[i, T:] == 0)
    assert torch.allclose(wav_percents, torch.from_numpy(z["wav_percents"]), atol=1e-7) and wav_percents.dtype == torch.float32
    assert texts.shape == (3, 11) and torch.equal(langs, torch.LongTensor([2, 0, 1])) and paths == ["f0.wav", "f1.wav", "f2.wav"]
    assert torch.allclose(text_percents, torch.FloatTensor([5 / 11, 8 / 11, 1.0]))
    # training flavour: the masks come from torch's default generator, like spectrogram_augment
    torch.manual_seed(42)
    tw = lid.DeviceCollate(fe, lang2index, train=True, mask_times=2)(batch)[0].cpu()
    torch.manual_seed(42)
    frames = [O.kaldi_num_frames(b[0].shape[-1]) for b in batch]
    m = lid.draw_masks(frames, 80, 0.05, 27, 2)
    for i in range(3):
        bounds = [tuple(int(v) for v in m[i, q]) for q in range(2)]
        ref = O.apply_mask_bounds(wavs[i, :frames[i]].cpu().T.unsqueeze(0), bounds)[0].T
        assert torch.equal(tw[i, :frames[i]], ref)


def test_resampler_matches_reference_data_processor(lid, golden_dir):
    """Row f4: the polyphase resampling kernel against the reference's DataProcessor outputs (golden) and against the
    oracle for other rate pairs (down- and up-sampling).  fp32 FIR of up to 475 taps in a different summation order:
    1e-5 absolute on signals of unit scale."""
    z = np.load(os.path.join(golden_dir, "resample.npz"))
    for rate, n in ((44100, 3), (22050, 4)):
        rs = lid.Resampler(rate, 16000)
        xs = [torch.from_numpy(z["in_%d_%d" % (rate, i)]) for i in range(n)]
        ys = rs.data_processor(xs)
        for i in range(n):
            want = torch.from_numpy(z["out_%d_%d" % (rate, i)])
            assert ys[i].is_cuda and ys[i].shape == want.shape, (rate, i, ys[i].shape, want.shape)
            assert torch.allclose(ys[i].cpu(), want, rtol=0, atol=1e-5), (rate, i, (ys[i].cpu() - want).abs().max())
    g = torch.Generator().manual_seed(5)
    for orig in (48000, 8000, 11025, 44100):
        rs = lid.Resampler(orig, 16000)
        xs = [torch.randn(n, generator=g) for n in (orig // 2 + 17, 999, 1)]
        ys = rs.resample_list(xs)
        for x, y in zip(xs, ys):
            want = O.resample(x, orig, 16000)
            assert y.shape == want.shape == (rs.out_len(x.numel()),)
            assert torch.allclose(y.cpu(), want, rtol=0, atol=1e-5), (orig, x.numel(), (y.cpu() - want).abs().max())
    same = lid.Resampler(16000, 16000).resample_list([xs[0]])[0]
    assert torch.equal(same.cpu(), xs[0])
    # resampled audio feeds the front-end: 44.1 kHz in, 16 kHz fbank out
    rs = lid.Resampler(44100, 16000)
    x = torch.randn(44100, generator=g)
    y = rs.resample_list([x])[0]
    feats, _ = lid.FrontEnd(n_mels=80).featurize([y])
    want = O.kaldi_fbank(O.resample(x, 44100, 16000))
    _check_fbank(feats[0].cpu(), want, "resample -> fbank")
