"""CPU restatement of the speech-lid front-end (torch CPU ops, fp32).  TEST INFRASTRUCTURE ONLY.

Every function names the reference lines it follows.  ``ref:`` paths are relative to the
reference tree (kouyt5/speech-lid); ``ta:`` paths are relative to the torchaudio package the
reference calls into (pinned by the reference to 0.12.1, ``lid/requirements/install.sh:4``;
2.11.0 in this image), because that is where the arithmetic of this path lives.

The restatement uses the same torch CPU primitives in the same order as the reference path
(``torch.fft.rfft``, ``abs().pow(2)``, ``torch.mm`` ...), so on the same machine it is
bit-identical to ``lid.audio_processor`` -- ``tests/test_oracle_golden.py`` pins that against
``tests/golden/*.npz`` (outputs of the reference itself) and, when torchaudio is importable,
against ``torchaudio.compliance.kaldi`` live.

Not product code: the product package never imports this module.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import torch

EPS32 = float(torch.finfo(torch.float32).eps)  # ta: compliance/kaldi.py:22  (1.1920929e-07)


# --------------------------------------------------------------------------------------
# A1  normalize_wav                                   ref: lid/audio_processor.py:108-115
# --------------------------------------------------------------------------------------
def normalize_wav(wav: torch.Tensor) -> torch.Tensor:
    """(wav - mean) / (std + 1e-6), unbiased std over the last dim."""
    std, mean = torch.std_mean(wav, dim=-1)
    return torch.div(wav - mean, std + 1e-6)


# --------------------------------------------------------------------------------------
# A2  wav_augment: dither + 0.97 pre-emphasis         ref: lid/audio_processor.py:125-134
# (sox speed/pitch :135-154 and WavAugment reverb :155-163 are off-path: they need sox /
#  the `augment` package, neither of which exists in this image)
# --------------------------------------------------------------------------------------
def wav_dither_preemph(wav: torch.Tensor, noise: Optional[torch.Tensor] = None,
                       dither: float = 1e-5, coeff: float = 0.97) -> torch.Tensor:
    """``wav += 1e-5 * U[0,1)`` then ``y[0]=x[0]; y[n]=x[n]-0.97*x[n-1]``.

    ``noise`` is the U[0,1) draw (``torch.rand_like(wav)`` in the reference, CPU default
    generator); pass it explicitly to compare with a device implementation.  Unlike the
    reference this does NOT mutate ``wav`` in place (the reference does, ``:129``)."""
    if noise is None:
        noise = torch.rand_like(wav)
    wav = wav + dither * noise
    return torch.cat((wav[:, 0].unsqueeze(1), wav[:, 1:] - coeff * wav[:, :-1]), dim=1)


# --------------------------------------------------------------------------------------
# Tables                                                ta: compliance/kaldi.py:86-113,436-511
# --------------------------------------------------------------------------------------
def povey_window(n: int) -> torch.Tensor:
    """hann(n, periodic=False) ** 0.85                  ta: compliance/kaldi.py:98-100"""
    return torch.hann_window(n, periodic=False, dtype=torch.float32).pow(0.85)


def kaldi_mel_banks(num_bins: int, padded: int, sample_freq: float,
                    low_freq: float = 20.0, high_freq: float = 0.0) -> torch.Tensor:
    """Triangular banks on the 1127*ln(1+f/700) scale, (num_bins, padded/2 + 1) with the Nyquist
    column zero (vtln_warp == 1 branch).                ta: compliance/kaldi.py:436-511,621-630"""
    assert num_bins > 3 and padded % 2 == 0
    num_fft_bins = padded / 2
    nyquist = 0.5 * sample_freq
    if high_freq <= 0.0:
        high_freq += nyquist
    assert 0.0 <= low_freq < nyquist and 0.0 < high_freq <= nyquist and low_freq < high_freq
    fft_bin_width = sample_freq / padded
    mel_lo = 1127.0 * math.log(1.0 + low_freq / 700.0)
    mel_hi = 1127.0 * math.log(1.0 + high_freq / 700.0)
    delta = (mel_hi - mel_lo) / (num_bins + 1)
    b = torch.arange(num_bins).unsqueeze(1)
    left = mel_lo + b * delta
    center = mel_lo + (b + 1.0) * delta
    right = mel_lo + (b + 2.0) * delta
    mel = (1127.0 * (1.0 + (fft_bin_width * torch.arange(num_fft_bins)) / 700.0).log()).unsqueeze(0)
    up = (mel - left) / (center - left)
    down = (right - mel) / (right - center)
    banks = torch.max(torch.zeros(1), torch.min(up, down))
    return torch.nn.functional.pad(banks, (0, 1), mode="constant", value=0)


def kaldi_dct_matrix(num_ceps: int, num_mel_bins: int) -> torch.Tensor:
    """(num_mel_bins, num_ceps) DCT-II ortho with column 0 = sqrt(1/num_mel_bins).
    ta: compliance/kaldi.py:648-658 over ta: functional/functional.py:636-667"""
    n = torch.arange(float(num_mel_bins))
    k = torch.arange(float(num_mel_bins)).unsqueeze(1)
    dct = torch.cos(math.pi / float(num_mel_bins) * (n + 0.5) * k)
    dct[0] *= 1.0 / math.sqrt(2.0)
    dct *= math.sqrt(2.0 / float(num_mel_bins))
    dct = dct.t()  # keep the transposed view: the reference's matmul sees this memory layout
    dct[:, 0] = math.sqrt(1 / float(num_mel_bins))
    return dct[:, :num_ceps]


def kaldi_lifter(num_ceps: int, cepstral_lifter: float) -> torch.Tensor:
    """1 + 0.5*L*sin(pi*i/L)                            ta: compliance/kaldi.py:661-666"""
    i = torch.arange(num_ceps)
    return 1.0 + 0.5 * cepstral_lifter * torch.sin(math.pi * i / cepstral_lifter)


# --------------------------------------------------------------------------------------
# Framing                                               ta: compliance/kaldi.py:44-83,154-217
# --------------------------------------------------------------------------------------
def kaldi_window(window_type: str, n: int, blackman_coeff: float = 0.42) -> torch.Tensor:
    """The five windows of ``_feature_window_function``.          ta: compliance/kaldi.py:86-113"""
    if window_type == "povey":
        return povey_window(n)
    if window_type == "hanning":
        return torch.hann_window(n, periodic=False, dtype=torch.float32)
    if window_type == "hamming":
        return torch.hamming_window(n, periodic=False, alpha=0.54, beta=0.46, dtype=torch.float32)
    if window_type == "rectangular":
        return torch.ones(n, dtype=torch.float32)
    if window_type == "blackman":
        a = 2 * math.pi / (n - 1)
        w = torch.arange(n, dtype=torch.float32)
        return (blackman_coeff - 0.5 * torch.cos(a * w) + (0.5 - blackman_coeff) * torch.cos(2 * a * w)).to(torch.float32)
    raise Exception("Invalid window type " + window_type)


def kaldi_num_frames(num_samples: int, window_size: int = 400, window_shift: int = 160) -> int:
    """snip_edges=True frame count; 0 when the utterance is shorter than one window.
    ta: compliance/kaldi.py:63-67"""
    if num_samples < window_size:
        return 0
    return 1 + (num_samples - window_size) // window_shift


def kaldi_windowed_frames(wav1d: torch.Tensor, window_size: int, window_shift: int, padded: int,
                          preemph: float, remove_dc: bool = True, window_type: str = "povey") -> torch.Tensor:
    """(m, padded) windowed, zero-padded frames.        ta: compliance/kaldi.py:154-217"""
    n = wav1d.numel()
    # ta: compliance/kaldi.py:142  (the reference inherits this assertion; N < window raises)
    assert 2 <= window_size <= n, "choose a window size {} that is [2, {}]".format(window_size, n)
    m = kaldi_num_frames(n, window_size, window_shift)
    wav1d = wav1d.contiguous()
    frames = wav1d.as_strided((m, window_size), (window_shift, 1))
    if remove_dc:
        frames = frames - torch.mean(frames, dim=1).unsqueeze(1)
    if preemph != 0.0:
        shifted = torch.nn.functional.pad(frames.unsqueeze(0), (1, 0), mode="replicate").squeeze(0)
        frames = frames - preemph * shifted[:, :-1]
    frames = frames * kaldi_window(window_type, window_size).unsqueeze(0)
    if padded != window_size:
        frames = torch.nn.functional.pad(frames.unsqueeze(0), (0, padded - window_size),
                                         mode="constant", value=0).squeeze(0)
    return frames


# --------------------------------------------------------------------------------------
# A4  kaldi fbank as the reference calls it             ref: lid/audio_processor.py:41-69
#                                                       ta: compliance/kaldi.py:514-645
# --------------------------------------------------------------------------------------
def kaldi_fbank(wav: torch.Tensor, n_mels: int = 80, sr: int = 16000, frame_length_ms: int = 25,
                frame_shift_ms: int = 10, preemph: float = 1.0, window_type: str = "povey",
                remove_dc: bool = True) -> torch.Tensor:
    """(1,N) or (N,) fp32 -> (m, n_mels) log-mel; dither 0, povey, remove_dc, snip_edges, power,
    low_freq 20, high_freq Nyquist -- the argument set of ``_kaidi_wav2mel``."""
    if wav.dim() == 2:
        wav = wav[0]  # channel=-1 -> channel 0          ta: compliance/kaldi.py:135-137
    shift = int(sr * frame_shift_ms * 0.001)
    size = int(sr * frame_length_ms * 0.001)
    padded = 1 if size == 0 else 2 ** (size - 1).bit_length()
    frames = kaldi_windowed_frames(wav.to(torch.float32), size, shift, padded, preemph, remove_dc, window_type)
    spectrum = torch.fft.rfft(frames).abs().pow(2.0)
    banks = kaldi_mel_banks(n_mels, padded, float(sr))
    mel = torch.mm(spectrum, banks.T)
    return torch.max(mel, torch.tensor(EPS32)).log()


def wav2mel_kaldi(x: torch.Tensor, win_length: float = 0.025, hop_length: float = 0.01,
                  n_mels: int = 80, sr: int = 16000) -> torch.Tensor:
    """``wav2mel(x, use_kaildi=True)``: (1,N) -> (1, n_mels, T).  ref: lid/audio_processor.py:8-69"""
    f = kaldi_fbank(x, n_mels=n_mels, sr=sr, frame_length_ms=int(1000 * win_length),
                    frame_shift_ms=int(1000 * hop_length), preemph=1.0)
    return f.transpose(0, 1).unsqueeze(0)


# --------------------------------------------------------------------------------------
# A9  the reference's DEFAULT branch: MelSpectrogram + AmplitudeToDB(top_db=80)
#                                                       ref: lid/audio_processor.py:72-105
#     ta: transforms/_transforms.py (Spectrogram, MelScale, AmplitudeToDB), functional/functional.py:54-146,
#         :356-403 (amplitude_to_DB), :425-588 (_hz_to_mel, _mel_to_hz, melscale_fbanks)
# --------------------------------------------------------------------------------------
def htk_mel_fbanks(n_freqs: int, f_min: float, f_max: float, n_mels: int, sample_rate: int) -> torch.Tensor:
    """(n_freqs, n_mels) triangular filters on the HTK scale 2595*log10(1+f/700), norm=None.
    ta: functional/functional.py:492-588"""
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    m_min = 2595.0 * math.log10(1.0 + (f_min / 700.0))
    m_max = 2595.0 * math.log10(1.0 + (f_max / 700.0))
    m_pts = torch.linspace(m_min, m_max, n_mels + 2)
    f_pts = 700.0 * (10.0 ** (m_pts / 2595.0) - 1.0)
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    down = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up = slopes[:, 2:] / f_diff[1:]
    return torch.max(torch.zeros(1), torch.min(down, up))


def num_frames_centered(num_samples: int, hop: int = 160, pad: int = 0) -> int:
    """torch.stft(center=True): 1 + (N + 2*pad) // hop"""
    return 1 + (num_samples + 2 * pad) // hop


def melspec_db(x: torch.Tensor, win_length: float = 0.025, hop_length: float = 0.01, n_mels: int = 80,
               n_fft: int = 512, pad: int = 0, sr: int = 16000, top_db: Optional[float] = 80.0) -> torch.Tensor:
    """``wav2mel(x, use_kaildi=False)``: (1,N) -> (1, n_mels, 1 + (N+2*pad)//hop).  Note the reference does not forward
    ``sr`` to MelSpectrogram's mel scale (always 16 kHz): kept."""
    win = int(sr * win_length)
    hop = int(sr * hop_length)
    if pad > 0:
        x = torch.nn.functional.pad(x, (pad, pad), "constant")
    window = torch.hann_window(win)
    spec = torch.stft(input=x, n_fft=n_fft, hop_length=hop, win_length=win, window=window, center=True,
                      pad_mode="reflect", normalized=False, onesided=True, return_complex=True)
    spec = spec.abs().pow(2.0)                                                   # (1, n_fft/2+1, T)
    fb = htk_mel_fbanks(n_fft // 2 + 1, 0.0, float(16000 // 2), n_mels, 16000)
    mel = torch.matmul(spec.transpose(-1, -2), fb).transpose(-1, -2)             # (1, n_mels, T)
    db = 10.0 * torch.log10(torch.clamp(mel, min=1e-10))
    db -= 10.0 * math.log10(max(1e-10, 1.0))
    if top_db is not None:
        db = torch.max(db, (db.amax(dim=(-3, -2, -1)) - top_db).view(-1, 1, 1))
    return db


# --------------------------------------------------------------------------------------
# A5  MFCC (not in the reference; pinned to torchaudio.compliance.kaldi.mfcc with A4's framing)
#                                                       ta: compliance/kaldi.py:669-813
# --------------------------------------------------------------------------------------
def kaldi_mfcc(wav: torch.Tensor, num_ceps: int = 40, n_mels: int = 80, sr: int = 16000,
               cepstral_lifter: float = 22.0, preemph: float = 1.0) -> torch.Tensor:
    feat = kaldi_fbank(wav, n_mels=n_mels, sr=sr, preemph=preemph)
    feat = feat.matmul(kaldi_dct_matrix(num_ceps, n_mels))
    if cepstral_lifter != 0.0:
        feat *= kaldi_lifter(num_ceps, cepstral_lifter).unsqueeze(0).to(torch.float32)
    return feat


# --------------------------------------------------------------------------------------
# A6  SpecAugment                                       ref: lid/audio_processor.py:198-228
#                                                       ta: functional/functional.py:806-811,885-958
# --------------------------------------------------------------------------------------
def draw_mask_bounds(T: int, n_mels: int, t_mask: float = 0.05, f_mask: float = 27,
                     mask_times: int = 0, generator: Optional[torch.Generator] = None
                     ) -> List[Tuple[int, int, int, int]]:
    """Integer (t0, t1, f0, f1) per mask iteration, consuming the CPU RNG exactly as
    ``TimeMasking(int(T*t_mask))`` then ``FrequencyMasking(f_mask)`` do: two ``torch.rand(1)``
    per mask, none when the mask parameter is < 1."""
    out = []
    for _ in range(mask_times):
        b = []
        for axis_len, param in ((T, int(T * t_mask)), (n_mels, f_mask)):
            if param < 1:
                b += [0, 0]
                continue
            value = torch.rand(1, generator=generator) * param
            min_value = torch.rand(1, generator=generator) * (axis_len - value)
            start = int(min_value.long())
            end = start + int(value.long())
            if end - start >= param:  # ta: functional/functional.py:948-949
                raise ValueError("Number of columns to be masked should be less than mask_param")
            b += [start, end]
        out.append(tuple(b))
    return out


def apply_mask_bounds(spec: torch.Tensor, bounds: Sequence[Sequence[int]]) -> torch.Tensor:
    """spec (1, n_mels, T) -> copy with [t0,t1) columns and [f0,f1) rows set to 0.0
    (mask_value=0.0, ta: transforms/_transforms.py _AxisMasking.forward)."""
    spec = spec.clone()
    for t0, t1, f0, f1 in bounds:
        spec[..., :, t0:t1] = 0.0
        spec[..., f0:f1, :] = 0.0
    return spec


def spectrogram_augment(spec: torch.Tensor, t_mask: float = 0.05, f_mask: float = 27,
                        mask_times: int = 0, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """t_stretch=False branch of ``spectrogram_augment``; spec is (1, n_mels, T)."""
    bounds = draw_mask_bounds(spec.size(2), spec.size(1), t_mask, f_mask, mask_times, generator)
    return apply_mask_bounds(spec, bounds)


# --------------------------------------------------------------------------------------
# A7  CMVN -- NOT on the reference hot path (commented out at ref: lid/audio_processor.py:66-68,
#     lid/conformer.py:314-315).  OUR definition; parity unpinned.
# --------------------------------------------------------------------------------------
CMVN_EPS = 1e-9  # the epsilon in the reference's commented-out line (audio_processor.py:68)


def cmvn_per_utt(feat: torch.Tensor) -> torch.Tensor:
    """feat (T, D) fp32 -> per-dimension (x - mean_t) / (std_t + 1e-9), unbiased std, statistics
    in fp64 over the utterance's own frames, result rounded to fp32."""
    x = feat.double()
    std, mean = torch.std_mean(x, dim=0)
    return ((x - mean) / (std + CMVN_EPS)).float()


def cmvn_stats(feats: Sequence[torch.Tensor]) -> torch.Tensor:
    """[sum_d (D), sumsq_d (D), count] in fp64 over all frames of all (T_i, D) tensors -- the
    vector each rank all-reduces for global CMVN."""
    D = feats[0].shape[1]
    s = torch.zeros(2 * D + 1, dtype=torch.float64)
    for f in feats:
        x = f.double()
        s[:D] += x.sum(0)
        s[D:2 * D] += (x * x).sum(0)
        s[2 * D] += x.shape[0]
    return s


def cmvn_finalize(stats: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """stats [2D+1] fp64 -> (mean (D), unbiased std (D)) fp64."""
    D = (stats.numel() - 1) // 2
    n = stats[2 * D]
    mean = stats[:D] / n
    var = (stats[D:2 * D] - stats[:D] * mean) / (n - 1.0)
    return mean, var.clamp_min(0.0).sqrt()


def cmvn_apply(feat: torch.Tensor, mean: torch.Tensor, std: torch.Tensor) -> torch.Tensor:
    return ((feat.double() - mean) / (std + CMVN_EPS)).float()


# --------------------------------------------------------------------------------------
# A8  feature contract                                  ref: lid/raw_datasets.py:345-365
# --------------------------------------------------------------------------------------
def collate_features(specs: Sequence[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
    """specs: list of (1, D, T_i) -> (wavs (B, T_max, D) zero padded, wav_percents (B,) = T_i/T_max)."""
    rows = [s.squeeze(0).transpose(0, 1) for s in specs]
    wavs = torch.nn.utils.rnn.pad_sequence(rows, batch_first=True)
    percents = torch.tensor([r.shape[0] / wavs.shape[1] for r in rows], dtype=torch.float32)
    return wavs, percents


# --------------------------------------------------------------------------------------
# fp64 "truth" with the oracle's fp32 tables (SURVEY.md appendix A.3): calibrates tolerances.
# --------------------------------------------------------------------------------------
def truth64_fbank(wav: torch.Tensor, n_mels: int = 80, preemph: float = 1.0, window_type: str = "povey",
                  remove_dc: bool = True, in_scale: float = 1.0) -> torch.Tensor:
    """``kaldi_fbank`` in float64 on the same fp32 tables: (m, n_mels).  ``in_scale`` multiplies the samples first
    (int16 PCM); it is rounded to fp32, as the front-end's configuration holds it, and the product is exact in fp64."""
    if wav.dim() == 2:
        wav = wav[0]
    w = wav.double() * float(torch.tensor(in_scale, dtype=torch.float32))
    m = kaldi_num_frames(w.numel())
    idx = torch.arange(m)[:, None] * 160 + torch.arange(400)[None]
    fr = w[idx]
    if remove_dc:
        fr = fr - fr.mean(1, keepdim=True)
    if preemph != 0.0:
        fr = fr - preemph * torch.cat([fr[:, :1], fr[:, :-1]], 1)
    fr = torch.nn.functional.pad(fr * kaldi_window(window_type, 400).double(), (0, 112))
    X = torch.fft.rfft(fr)
    mel = (X.real ** 2 + X.imag ** 2) @ kaldi_mel_banks(n_mels, 512, 16000.0).double().T
    return mel.clamp_min(EPS32).log()


def truth64_melspec_db(x: torch.Tensor, pad: int = 0, top_db: Optional[float] = 80.0, n_mels: int = 80) -> torch.Tensor:
    """``melspec_db`` -- the reference's default branch (ref: lid/audio_processor.py:72-105 -> torch.stft(center=True,
    reflect), HTK mel, AmplitudeToDB(top_db)) -- in float64 on the fp32 tables: (T, n_mels).  ``top_db=None``: no clamp."""
    w = x.reshape(-1).double()
    if pad:
        w = torch.nn.functional.pad(w, (pad, pad))
    wp = torch.nn.functional.pad(w[None, None], (256, 256), mode="reflect")[0, 0]
    T = 1 + w.numel() // 160
    fr = wp[torch.arange(T)[:, None] * 160 + torch.arange(512)[None]]
    win = torch.zeros(512, dtype=torch.float64)
    win[56:456] = torch.hann_window(400).double()
    X = torch.fft.rfft(fr * win)
    mel = (X.real ** 2 + X.imag ** 2) @ htk_mel_fbanks(257, 0.0, 8000.0, n_mels, 16000).double()
    db = 10.0 * torch.log10(mel.clamp_min(1e-10))
    if top_db is None:
        return db
    return torch.maximum(db, db.max() - top_db)


def truth64_resample(x: torch.Tensor, kernel32: torch.Tensor, width: int, orig: int, new: int) -> torch.Tensor:
    """``resample`` of one utterance in float64 on the fp32 FIR bank ``kernel32`` ((new/g, 2 width + orig/g), g the gcd):
    output sample i * new + p is  sum_k kernel32[p][k] * xpad[i * orig + k],  xpad = x with ``width`` zeros in front and
    width + orig behind, cut to ceil(new * n / orig) samples.  Runs on x's device."""
    g = math.gcd(int(orig), int(new))
    orig, new = int(orig) // g, int(new) // g
    w = x.reshape(-1).double()
    k = kernel32.to(w.device).double()
    assert k.shape[0] == new and k.shape[1] == 2 * width + orig
    xp = torch.nn.functional.pad(w, (width, width + orig))
    y = (xp.unfold(0, k.shape[1], orig) @ k.T).reshape(-1)
    return y[:-(-new * w.numel() // orig)]


def truth64_s3prl_fbank(x: torch.Tensor, fbank_size: int = 80, n_fft: int = 640, normalize: bool = True) -> torch.Tensor:
    """``s3prl_fbank`` in float64 on the reference's fp32 tables (``torch.hann_window(n_fft)``, ``melscale_fbanks``):
    spectrogram (center=False, hop n_fft / 2, power 2) -> HTK mel -> 10 log10(max(., 1e-10)) -> (x - mean) / (std + 1e-9)
    with one mean / unbiased std over the whole spectrogram.  (frames, fbank_size), on x's device."""
    w = x.reshape(-1).double()
    window = torch.hann_window(n_fft).double().to(w.device)
    spec = torch.stft(w, n_fft=n_fft, hop_length=n_fft // 2, win_length=n_fft, window=window, center=False,
                      normalized=False, onesided=True, return_complex=True)
    power = spec.real ** 2 + spec.imag ** 2                                      # (n_fft/2+1, frames)
    fb = htk_mel_fbanks(n_fft // 2 + 1, 0.0, 8000.0, fbank_size, 16000).double().to(w.device)
    db = 10.0 * torch.log10((power.T @ fb).clamp_min(1e-10))
    if not normalize:
        return db
    std, mean = torch.std_mean(db)
    return (db - mean) / (std + 1e-9)


# --------------------------------------------------------------------------------------
# Synthetic inputs (SURVEY.md §8d).  Deterministic; used by tests, golden generation and bench.
# --------------------------------------------------------------------------------------
def synth_noise(n: int, seed: int) -> torch.Tensor:
    """normalize_wav(randn(1, n)) from torch.Generator().manual_seed(seed)."""
    g = torch.Generator().manual_seed(seed)
    return normalize_wav(torch.randn(1, n, generator=g))


def synth_speechlike(n: int, seed: int) -> torch.Tensor:
    """Harmonic stack sum_k sin(2 pi k f0 t)/k (f0~U(90,250), k<=40) + 1/f-shaped noise at -30 dB."""
    g = torch.Generator().manual_seed(seed)
    f0 = 90.0 + 160.0 * float(torch.rand(1, generator=g))
    t = torch.arange(n, dtype=torch.float64) / 16000.0
    x = torch.zeros(n, dtype=torch.float64)
    for k in range(1, 41):
        if k * f0 < 8000.0:
            x += torch.sin(2 * math.pi * k * f0 * t) / k
    white = torch.randn(n, generator=g, dtype=torch.float64)
    spec = torch.fft.rfft(white)
    spec[1:] /= torch.sqrt(torch.arange(1, spec.numel(), dtype=torch.float64))
    pink = torch.fft.irfft(spec, n=n)
    pink *= (x.std() / pink.std()) * 10 ** (-30 / 20)
    return normalize_wav((x + pink).float().unsqueeze(0))


# --------------------------------------------------------------------------------------
# f4  resampling DataProcessor                          ref: lid/ConformerLangModel.py:131-178
#                                                       ta: functional/functional.py _get_sinc_resample_kernel,
#                                                           _apply_sinc_resample_kernel; transforms Resample
# --------------------------------------------------------------------------------------
def sinc_resample_kernel(orig_freq: int, new_freq: int, lowpass_filter_width: int = 6, rolloff: float = 0.99):
    import math
    g = math.gcd(int(orig_freq), int(new_freq))
    orig, new = int(orig_freq) // g, int(new_freq) // g
    base_freq = min(orig, new) * rolloff
    width = math.ceil(lowpass_filter_width * orig / base_freq)
    idx = torch.arange(-width, width + orig, dtype=torch.float64)[None, None] / orig
    t = torch.arange(0, -new, -1, dtype=None)[:, None, None] / new + idx
    t *= base_freq
    t = t.clamp_(-lowpass_filter_width, lowpass_filter_width)
    window = torch.cos(t * math.pi / lowpass_filter_width / 2) ** 2
    t *= math.pi
    kernels = torch.where(t == 0, torch.tensor(1.0).to(t), t.sin() / t)
    kernels *= window * (base_freq / orig)
    return kernels.to(torch.float32), width, orig, new


def resample(wav: torch.Tensor, orig_freq: int, new_freq: int = 16000) -> torch.Tensor:
    """(N,) or (B, N) fp32 -> resampled, as torchaudio.transforms.Resample(orig_freq, new_freq) with its defaults."""
    if orig_freq == new_freq:
        return wav
    kernel, width, orig, new = sinc_resample_kernel(orig_freq, new_freq)
    shape = wav.shape
    x = wav.reshape(-1, shape[-1])
    length = x.shape[1]
    x = torch.nn.functional.pad(x, (width, width + orig))
    y = torch.nn.functional.conv1d(x[:, None], kernel, stride=orig)
    y = y.transpose(1, 2).reshape(x.shape[0], -1)
    target = int(torch.ceil(torch.as_tensor(new * length / orig)).long())
    return y[..., :target].reshape(shape[:-1] + (target,))


def data_processor(x: Sequence[torch.Tensor], sample_rate: int) -> Sequence[torch.Tensor]:
    """DataProcessor.forward (ref: lid/ConformerLangModel.py:146-169)."""
    if sample_rate not in (22050, 44100):
        return x
    longest = max(int(w.shape[-1]) for w in x)
    percent = [int(w.shape[-1]) / longest for w in x]
    padded = torch.nn.utils.rnn.pad_sequence(list(x), batch_first=True)
    y = resample(padded, sample_rate, 16000)
    lens = [int(p * y.shape[-1]) for p in percent]
    return [y[i, :lens[i]] for i in range(len(lens))]


# --------------------------------------------------------------------------------------
# f4b  the wav2vec-exp FBank variant                      ref: wav2vec-exp/s3prl_model.py:174-204
#      F.spectrogram(pad=0, hann_window(n_fft), n_fft, hop=n_fft//2, win=n_fft, power=2, center=False)
#      -> HTK mel (f_max 8000, norm=None) -> amplitude_to_DB(10, amin=1e-10, db_multiplier=0, top_db=None)
#      -> (spec - mean) / (std + 1e-9) with ONE mean / unbiased std over the whole (n_mels, T) spectrogram
#      ta: functional/functional.py:54-146 (spectrogram), :356-403 (amplitude_to_DB), :492-588 (melscale_fbanks)
# --------------------------------------------------------------------------------------
def s3prl_fbank_num_frames(num_samples: int, n_fft: int = 640) -> int:
    """torch.stft(center=False): 1 + (N - n_fft) // hop, hop = n_fft // 2"""
    return 1 + (num_samples - n_fft) // (n_fft // 2) if num_samples >= n_fft else 0


def s3prl_fbank(x: torch.Tensor, fbank_size: int = 80, n_fft: int = 640, normalize: bool = True) -> torch.Tensor:
    """(T,) -> (fbank_size, frames), as ``FBank.forward`` (ref: wav2vec-exp/s3prl_model.py:181-204)."""
    fb = htk_mel_fbanks(n_fft // 2 + 1, 0.0, 8000.0, fbank_size, 16000)
    window = torch.hann_window(n_fft)
    spec = torch.stft(input=x.reshape(-1, x.shape[-1]), n_fft=n_fft, hop_length=n_fft // 2, win_length=n_fft, window=window,
                      center=False, pad_mode="reflect", normalized=False, onesided=True, return_complex=True)
    spec = spec.reshape(x.shape[:-1] + spec.shape[-2:]).abs().pow(2.0).float()     # (n_fft/2+1, T)
    spec = torch.matmul(spec.transpose(-1, -2), fb).transpose(-1, -2).float()
    spec = (10.0 * torch.log10(torch.clamp(spec, min=1e-10))).float()
    if not normalize:
        return spec
    std, mean = torch.std_mean(spec)
    return (spec - mean) / (std + 1e-9)
