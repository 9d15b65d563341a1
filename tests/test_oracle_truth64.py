"""CPU pins of the fp64 references (oracle.frontend_oracle.truth64_fbank / truth64_melspec_db) that
tests/test_gpu_dispatch.py holds every feature-kernel route to.  On speech-like input, where the fp32 oracle is itself
accurate, each fp64 reference must lie within fp32 distance of the fp32 oracle of the same configuration, and each
argument must change the result (a reference that ignored one would pass every kernel bug behind it)."""
import math

import pytest
import torch

from oracle import frontend_oracle as O

FP32_DISTANCE = 5e-5        # norm-relative; the measured distances are 1e-7 .. 2e-5


def _norm_rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())


@pytest.fixture(scope="module")
def speech():
    return O.synth_speechlike(20000, 7)


def _truth64_fbank_before_generalisation(wav, n_mels=80, preemph=1.0):
    """truth64_fbank as it read before it took window_type / remove_dc / in_scale: its defaults must not move."""
    w = wav[0].double()
    m = O.kaldi_num_frames(w.numel())
    fr = w[torch.arange(m)[:, None] * 160 + torch.arange(400)[None]]
    fr = fr - fr.mean(1, keepdim=True)
    fr = fr - preemph * torch.cat([fr[:, :1], fr[:, :-1]], 1)
    fr = torch.nn.functional.pad(fr * O.povey_window(400).double(), (0, 112))
    X = torch.fft.rfft(fr)
    mel = (X.real ** 2 + X.imag ** 2) @ O.kaldi_mel_banks(n_mels, 512, 16000.0).double().T
    return mel.clamp_min(O.EPS32).log()


def test_truth64_fbank_defaults_unchanged(speech):
    noise = O.synth_noise(16000, 3)
    for x in (speech, noise):
        assert torch.equal(O.truth64_fbank(x), _truth64_fbank_before_generalisation(x))
        assert torch.equal(O.truth64_fbank(x, n_mels=40, preemph=0.97), _truth64_fbank_before_generalisation(x, 40, 0.97))


@pytest.mark.parametrize("window", ["povey", "hanning", "hamming", "rectangular", "blackman"])
@pytest.mark.parametrize("remove_dc,preemph,n_mels", [(True, 1.0, 80), (False, 0.97, 80), (True, 0.97, 40),
                                                      (True, 1.0, 64), (True, 0.97, 23)])
def test_truth64_fbank_is_the_oracle_in_fp64(speech, window, remove_dc, preemph, n_mels):
    tru = O.truth64_fbank(speech, n_mels=n_mels, preemph=preemph, window_type=window, remove_dc=remove_dc)
    ref = O.kaldi_fbank(speech, n_mels=n_mels, preemph=preemph, window_type=window, remove_dc=remove_dc)
    assert tru.dtype == torch.float64 and tru.shape == ref.shape
    assert _norm_rel(ref, tru) <= FP32_DISTANCE
    other = "hamming" if window == "povey" else "povey"
    assert _norm_rel(O.truth64_fbank(speech, n_mels=n_mels, preemph=preemph, window_type=other, remove_dc=remove_dc),
                     tru) > 1e-3


def test_truth64_fbank_remove_dc_and_in_scale():
    x = O.synth_speechlike(20000, 8) + 0.5                 # the DC offset is what remove_dc takes out
    kw = dict(preemph=0.97, window_type="hamming")
    for rd in (True, False):
        assert _norm_rel(O.kaldi_fbank(x, remove_dc=rd, **kw), O.truth64_fbank(x, remove_dc=rd, **kw)) <= FP32_DISTANCE
    assert _norm_rel(O.truth64_fbank(x, remove_dc=False, **kw), O.truth64_fbank(x, remove_dc=True, **kw)) > 1e-3
    pcm = (O.synth_speechlike(20000, 9) * 3000).round().clamp(-32768, 32767).to(torch.int16)
    for scale in (1.0 / 32768.0, 1.0 / 3000.0):
        tru = O.truth64_fbank(pcm, in_scale=scale)
        assert _norm_rel(O.kaldi_fbank(pcm.float() * scale), tru) <= FP32_DISTANCE
        # the scale is the fp32 value the front-end's configuration holds; the product is exact in fp64
        s32 = float(torch.tensor(scale, dtype=torch.float32))
        assert torch.equal(tru, O.truth64_fbank(pcm.double() * s32))
    assert not torch.equal(O.truth64_fbank(pcm, in_scale=1.0 / 3000.0), O.truth64_fbank(pcm, in_scale=1.0 / 32768.0))


@pytest.mark.parametrize("pad", [0, 2, 4, 8, 16, 300])
@pytest.mark.parametrize("top_db,n_mels", [(80.0, 80), (20.0, 80), (None, 80), (80.0, 64)])
def test_truth64_melspec_db_is_the_oracle_in_fp64(speech, pad, top_db, n_mels):
    tru = O.truth64_melspec_db(speech, pad=pad, top_db=top_db, n_mels=n_mels)
    ref = O.melspec_db(speech, pad=pad, top_db=top_db, n_mels=n_mels)[0].T
    assert tru.dtype == torch.float64 and tru.shape == ref.shape == (O.num_frames_centered(20000, pad=pad), n_mels)
    assert _norm_rel(ref, tru) <= FP32_DISTANCE
    if top_db is not None:
        assert float(tru.max() - tru.min()) <= top_db + 1e-9
        if top_db < 40:
            assert float(tru.min()) == float(tru.max()) - top_db      # the clamp bites on this input
    if pad:
        assert not torch.equal(tru, O.truth64_melspec_db(speech, pad=0, top_db=top_db, n_mels=n_mels)[:tru.shape[0]])


def test_truth64_melspec_db_silence_and_short_input():
    assert torch.equal(O.truth64_melspec_db(torch.zeros(1, 2560)), torch.full((17, 80), -100.0, dtype=torch.float64))
    x = torch.randn(1, 1, generator=torch.Generator().manual_seed(1))     # 1 + 2 * 300 > 256: one sample is legal
    tru = O.truth64_melspec_db(x, pad=300, top_db=None)
    assert tru.shape == (4, 80) and _norm_rel(O.melspec_db(x, pad=300, top_db=None)[0].T, tru) <= FP32_DISTANCE


@pytest.mark.parametrize("n_ceps,n_mels,preemph", [(40, 80, 1.0), (13, 23, 0.97), (60, 80, 1.0)])
def test_truth64_mfcc_is_the_oracle_in_fp64(speech, n_ceps, n_mels, preemph):
    tru = (O.truth64_fbank(speech, n_mels=n_mels, preemph=preemph) @ O.kaldi_dct_matrix(n_ceps, n_mels).double()
           ) * O.kaldi_lifter(n_ceps, 22.0).double()
    assert _norm_rel(O.kaldi_mfcc(speech, num_ceps=n_ceps, n_mels=n_mels, preemph=preemph), tru) <= FP32_DISTANCE
    assert math.isfinite(float(tru.abs().max()))


# ---- the windowed-GEMM family (tests/test_gpu_gemm_routes.py): resampler and wav2vec-exp FBank ------------------------
@pytest.mark.parametrize("orig,new", [(44100, 16000), (22050, 16000), (48000, 16000), (8000, 16000), (16000, 44100),
                                      (88200, 16000)])
def test_truth64_resample_is_the_oracle_in_fp64(speech, orig, new):
    kernel, width, _, _ = O.sinc_resample_kernel(orig, new)
    x = speech[0]
    tru = O.truth64_resample(x, kernel[:, 0], width, orig, new)
    ref = O.resample(x, orig, new)
    assert tru.dtype == torch.float64 and tru.shape == ref.shape
    assert _norm_rel(ref, tru) <= FP32_DISTANCE
    # torchaudio's formulation -- a strided conv1d of the padded waveform -- evaluated in float64
    g = math.gcd(orig, new)
    xp = torch.nn.functional.pad(x.double(), (width, width + orig // g))
    conv = torch.nn.functional.conv1d(xp[None, None], kernel.double(), stride=orig // g)[0].T.reshape(-1)[:tru.numel()]
    assert float((conv - tru).abs().max()) <= 1e-13 * float(tru.abs().max())
    # every argument matters: the bank, its width, each rate, and the samples themselves
    other_k, other_w, _, _ = O.sinc_resample_kernel(orig + 50, new)
    if other_k.shape[0] == kernel.shape[0] and other_k.shape[2] == kernel.shape[2]:
        assert _norm_rel(O.truth64_resample(x, other_k[:, 0], other_w, orig, new), tru) > 1e-6
    assert _norm_rel(O.truth64_resample(x, kernel[:, 0] * (1 + 1e-3), width, orig, new), tru) > 1e-4
    y = x.clone()
    y[len(y) // 2] += 1.0
    assert not torch.equal(O.truth64_resample(y, kernel[:, 0], width, orig, new), tru)
    with pytest.raises(AssertionError):              # a bank of another width or rate pair is refused, not misread
        O.truth64_resample(x, kernel[:, 0], width + 1, orig, new)
    with pytest.raises(AssertionError):
        O.truth64_resample(x, kernel[:, 0], width, orig, new * 2 + 1)
    assert O.truth64_resample(x[:1], kernel[:, 0], width, orig, new).numel() == -(-(new // g) // (orig // g))


@pytest.mark.parametrize("fbank_size,n_fft", [(80, 640), (80, 320), (40, 640), (128, 640), (1, 640), (80, 2048),
                                              (80, 64), (80, 4)])
def test_truth64_s3prl_fbank_is_the_oracle_in_fp64(speech, fbank_size, n_fft):
    x = speech[0]
    raw = O.truth64_s3prl_fbank(x, fbank_size, n_fft, False)
    norm = O.truth64_s3prl_fbank(x, fbank_size, n_fft, True)
    std, mean = torch.std_mean(raw)
    assert torch.equal(norm, (raw - mean) / (std + 1e-9))
    for tru, normalize in ((raw, False), (norm, True)):
        ref = O.s3prl_fbank(x, fbank_size, n_fft, normalize).T
        assert tru.dtype == torch.float64 and tru.shape == ref.shape == (O.s3prl_fbank_num_frames(x.numel(), n_fft),
                                                                         fbank_size)
        # normalising divides the dB values' fp32 error by their std: the distance scales with it
        dist = FP32_DISTANCE * (float(raw.abs().max() / std / norm.abs().max()) if normalize else 1.0)
        assert _norm_rel(ref, tru) <= dist, (normalize, _norm_rel(ref, tru), dist)
    if fbank_size > 1 and n_fft >= 64:
        assert _norm_rel(O.truth64_s3prl_fbank(x, fbank_size - 1 if fbank_size > 2 else 3, n_fft, False)[:, -1:],
                         raw[:, -1:]) > 1e-3
    if n_fft >= 64:
        other = O.truth64_s3prl_fbank(x, fbank_size, n_fft - 2, False)
        assert other.shape != raw.shape or _norm_rel(other, raw) > 1e-4
    if n_fft == 4:                      # three bins under 80 triangles: empty filters floor at exactly -100 dB
        assert bool((raw == -100.0).all(0).any())


def test_truth64_s3prl_fbank_silence_and_one_value():
    z = O.truth64_s3prl_fbank(torch.zeros(6400), 80, 640, False)
    assert torch.equal(z, torch.full((19, 80), -100.0, dtype=torch.float64))
    assert torch.equal(O.truth64_s3prl_fbank(torch.zeros(6400), 80, 640, True), torch.zeros(19, 80, dtype=torch.float64))
    one = O.truth64_s3prl_fbank(torch.randn(640, generator=torch.Generator().manual_seed(2)), 1, 640, True)
    assert one.shape == (1, 1) and bool(torch.isnan(one).all())            # torch.std of one value
    assert bool(torch.isnan(O.s3prl_fbank(torch.randn(640), 1, 640)).all())
