"""Additive noise at a per-utterance SNR, mixed on the device (``FrontEnd.add_noise``, ``lidfe_add_noise``).

The definition is ``torchaudio.functional.add_noise``: for utterance ``u`` with samples ``x`` and noise ``nu`` of the
same length, ``y = x + a * nu`` with ``a = sqrt(E_x / E_nu * 10^(-snr / 10))`` (energies in fp64).  The noise is a
window of a clip of a ``NoiseBank`` (the clip repeats when it is shorter than the utterance) or N(0,1) drawn on the
device from a Philox stream.  ``snr = +inf`` leaves an utterance clean; it is how a batch mixes clean and noisy
utterances.  This module holds the host side: the bank, the per-batch draw and its validation.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple, Union

import torch

Snr = Union[float, Tuple[float, float]]


class NoiseBank:
    """Noise clips concatenated into one float32 device tensor (``data``); ``offsets`` / ``lengths`` stay on the host.
    Every clip must be non-empty, finite and carry energy (an all-zero clip has no SNR)."""

    def __init__(self, clips: Sequence[torch.Tensor], device: Union[str, torch.device, None] = None):
        if len(clips) == 0:
            raise ValueError("a NoiseBank needs at least one clip")
        host, self.offsets, self.lengths, pos = [], [], [], 0
        for k, c in enumerate(clips):
            c = torch.as_tensor(c)
            if c.dim() == 2:
                c = c[0]        # first channel, as FrontEnd.pack does
            c = c.detach().to("cpu", torch.float32).reshape(-1)
            if c.numel() == 0:
                raise ValueError("noise clip %d is empty" % k)
            if not bool(torch.isfinite(c).all()):
                raise ValueError("noise clip %d has non-finite samples" % k)
            if float(c.double().square().sum()) == 0.0:
                raise ValueError("noise clip %d has zero energy" % k)
            host.append(c)
            self.offsets.append(pos)
            self.lengths.append(int(c.numel()))
            pos += int(c.numel())
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.data = torch.cat(host).to(self.device).contiguous()

    def __len__(self) -> int:
        return len(self.lengths)


@dataclass
class NoiseDraw:
    """Per-utterance noise of one batch, on the host: SNR in dB (float32, +inf = clean), the bank clip and the start
    inside it (int64; None for the Gaussian source), and the 64-bit key of the Gaussian Philox stream."""
    snr_db: torch.Tensor
    clip: Optional[torch.Tensor]
    start: Optional[torch.Tensor]
    seed: int

    @property
    def batch(self) -> int:
        return int(self.snr_db.numel())


def _snr_range(snr_db: Snr) -> Tuple[float, float]:
    if isinstance(snr_db, (tuple, list)):
        if len(snr_db) != 2:
            raise ValueError("snr_db must be a number or a (lo, hi) range")
        lo, hi = float(snr_db[0]), float(snr_db[1])
        if not (math.isfinite(lo) and math.isfinite(hi)):
            raise ValueError("an SNR range must be finite, got (%r, %r)" % (lo, hi))
        if lo > hi:
            raise ValueError("SNR range (%r, %r) has lo > hi" % (lo, hi))
        return lo, hi
    v = float(snr_db)
    if math.isnan(v) or v == -math.inf:
        raise ValueError("snr_db must not be NaN or -inf, got %r" % v)
    return v, v


def draw_noise(batch: int, snr_db: Snr, p: float = 1.0, bank: Optional[NoiseBank] = None,
               generator: Optional[torch.Generator] = None) -> NoiseDraw:
    """Draw the noise of ``batch`` utterances.  ``snr_db``: a number, or ``(lo, hi)`` for U[lo, hi) per utterance;
    with probability ``1 - p`` an utterance stays clean (SNR +inf).

    Draw order on ``generator`` (the global CPU generator when None), always all of it, so the stream advances by the
    same amount whatever ``p`` is: ``rand(batch, float64)`` for the keep test (``< p``), ``rand(batch, float64)`` for
    the SNR (``lo + (hi - lo) * u``, then float32); with a bank ``randint(len(bank), (batch,))`` for the clip and
    ``rand(batch, float64)`` for the start (``floor(u * clip length)``); last ``randint(0, 2**63 - 1, (1,))`` for the
    Gaussian seed."""
    B = int(batch)
    if B < 0:
        raise ValueError("batch must be >= 0")
    p = float(p)
    if not 0.0 <= p <= 1.0:
        raise ValueError("p must lie in [0, 1], got %r" % p)
    lo, hi = _snr_range(snr_db)
    keep = torch.rand(B, dtype=torch.float64, generator=generator) < p
    u = torch.rand(B, dtype=torch.float64, generator=generator)
    snr = (lo + (hi - lo) * u) if hi > lo else torch.full((B,), lo, dtype=torch.float64)
    snr = torch.where(keep, snr, torch.full_like(snr, math.inf)).to(torch.float32)
    clip = start = None
    if bank is not None:
        clip = torch.randint(len(bank), (B,), generator=generator, dtype=torch.int64)
        lens = torch.tensor(bank.lengths, dtype=torch.int64)[clip]
        s = torch.rand(B, dtype=torch.float64, generator=generator)
        start = torch.minimum((s * lens.double()).floor().to(torch.int64), lens - 1)
    seed = int(torch.randint(0, 2 ** 63 - 1, (1,), generator=generator, dtype=torch.int64))
    return NoiseDraw(snr_db=snr, clip=clip, start=start, seed=seed)


def noise_table(draw: NoiseDraw, bank: Optional[NoiseBank], batch: int):
    """Validate a draw against the batch and the bank -> (int64 [3, B] clip offset / length / start or None for the
    Gaussian source, float32 [B] SNR), host tensors ready for upload."""
    snr = torch.as_tensor(draw.snr_db).to(torch.float32).reshape(-1)
    if snr.numel() != batch:
        raise ValueError("the draw holds %d SNRs for a batch of %d" % (snr.numel(), batch))
    if bool(torch.isnan(snr).any()) or bool((snr == -math.inf).any()):
        raise ValueError("SNRs must not be NaN or -inf (+inf leaves an utterance clean)")
    if bank is None:
        return None, snr.contiguous()
    if draw.clip is None or draw.start is None:
        raise ValueError("a bank needs a draw with clips and starts (draw_noise(..., bank=bank))")
    clip = torch.as_tensor(draw.clip).to(torch.int64).reshape(-1)
    start = torch.as_tensor(draw.start).to(torch.int64).reshape(-1)
    if clip.numel() != batch or start.numel() != batch:
        raise ValueError("the draw's clips / starts do not match the batch of %d" % batch)
    if batch and (int(clip.min()) < 0 or int(clip.max()) >= len(bank)):
        raise ValueError("clip index out of range [0, %d)" % len(bank))
    off = torch.tensor(bank.offsets, dtype=torch.int64)[clip]
    lens = torch.tensor(bank.lengths, dtype=torch.int64)[clip]
    if bool((start < 0).any()) or bool((start >= lens).any()):
        raise ValueError("start outside its clip")
    return torch.stack([off, lens, start]).contiguous(), snr.contiguous()


class NoiseAugment:
    """Noise augmentation for ``FrontEnd.featurize`` / ``DeviceCollate``: every batch draws its noise with
    ``draw_noise(B, snr_db, p, bank, generator)``.  The draws come from the augmentation's own ``generator`` (a fresh
    ``torch.Generator()`` when None; seed it for a reproducible run), never from the global one, so SpecAugment's
    mask stream is the same with noise on or off.  ``normalize=True`` runs normalize_wav on the mixture."""

    def __init__(self, bank: Optional[NoiseBank], snr_db: Snr, p: float = 1.0,
                 generator: Optional[torch.Generator] = None, normalize: bool = False):
        _snr_range(snr_db)
        if not 0.0 <= float(p) <= 1.0:
            raise ValueError("p must lie in [0, 1], got %r" % p)
        self.bank, self.snr_db, self.p = bank, snr_db, float(p)
        self.generator = generator if generator is not None else torch.Generator()
        self.normalize = bool(normalize)

    def draw(self, batch: int) -> NoiseDraw:
        return draw_noise(batch, self.snr_db, self.p, self.bank, self.generator)
