"""Device-side drop-in for ``MergedDataset.collate_fn`` (ref: lid/raw_datasets.py:345-365).

The reference's loader either ships features computed per file in its workers (``data.feature.type: mel`` -> the
collate pads them to ``(B, T_max, n_mels)``) or raw waveforms (``type: wav`` -> a list).  ``DeviceCollate`` takes the
items of the ``wav`` flavour -- ``(wav, token_ids, path, lang)`` -- and returns exactly the 6-tuple of the ``mel``
flavour, with the features computed for the whole batch by the CUDA front-end:

    wavs (B, T_max, n_out) float32 on the GPU, zero padded      texts (B, L_max) int64
    wav_percents (B,) float32 = T_i / T_max                     text_percents (B,) float32 = L_i / (L_max + 1e-9)
    audio_paths list[str]                                       langs (B,) int64

It must run in the training process (a CUDA context does not survive the DataLoader's fork): call it at the top of
``common_loop`` on the list the loader yields with ``collate_fn=lambda b: b``, or hand it to a ``num_workers=0`` loader.
SpecAugment follows the reference: masks only when ``train`` and ``mask_times > 0``, drawn per utterance in batch order
from torch's default CPU generator (ref: lid/raw_datasets.py:279-292, lid/audio_processor.py:198-228).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch.nn.utils.rnn import pad_sequence

from .specaug import draw_masks


def collate_host_part(batch: Sequence[Tuple], lang2index: Dict[str, int]):
    """Everything of the reference's collate that is not features (ref: lid/raw_datasets.py:353-365)."""
    texts = pad_sequence([item[1] for item in batch]).transpose(1, 0)
    audio_paths = [item[2] for item in batch]
    text_percents = torch.FloatTensor([item[1].shape[-1] / (texts.shape[1] + 1e-9) for item in batch])
    langs = torch.LongTensor([lang2index[item[3]] for item in batch])
    return texts, text_percents, audio_paths, langs


class DeviceCollate:
    def __init__(self, frontend, lang2index: Dict[str, int], train: bool = False, t_mask: float = 0.05,
                 f_mask: int = 27, mask_times: int = 0, cmvn: str = "none", noise=None):
        """``noise``: a ``NoiseAugment`` mixed into the waveforms of training batches (``train=True``) only; its draws
        come from its own generator, so the SpecAugment masks are the same with noise on or off."""
        if noise is not None and frontend.in_dtype != torch.float32:
            raise ValueError("noise augmentation needs a float32 FrontEnd")
        self.frontend = frontend
        self.noise = noise
        self.lang2index = dict(lang2index)
        self.train = bool(train)
        self.t_mask, self.f_mask, self.mask_times = float(t_mask), int(f_mask), int(mask_times)
        self.cmvn = cmvn

    def __call__(self, batch: Sequence[Tuple]):
        if len(batch) == 0:
            raise ValueError("empty batch")
        wavs: List[torch.Tensor] = [item[0][0] if item[0].dim() == 2 else item[0] for item in batch]   # channel 0
        masks = None
        if self.train and self.mask_times > 0:
            # drawn inside featurize once the H2D copies of the waveforms are under way (same RNG consumption)
            def masks(frames):
                return draw_masks(frames, self.frontend.n_out, self.t_mask, self.f_mask, self.mask_times)
        feats, wav_percents = self.frontend.featurize(wavs, masks=masks, cmvn=self.cmvn, cache_plan=False,
                                                      noise=self.noise if self.train else None)
        texts, text_percents, audio_paths, langs = collate_host_part(batch, self.lang2index)
        return feats, texts, wav_percents.to(torch.float32).cpu(), text_percents, audio_paths, langs
