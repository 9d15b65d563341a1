"""speech_lid_b200 -- B200-native front-end for kouyt5/speech-lid's ``lid/audio_processor.py`` path.

Raw 16 kHz waveforms -> Kaldi log-mel fbank / MFCC -> SpecAugment masks -> CMVN -> ``(B, T, n_out)``
features, computed by hand-written sm_100a kernels behind a C ABI (``include/lidfe.h``).  There is no
CPU fallback: importing works anywhere, computing needs the built ``liblidfe.so`` and a GPU.
"""
from . import _lib, tables
from ._lib import LIB_PATH, LidfeError, load_library
from .collate import DeviceCollate, collate_host_part
from .frontend import FrontEnd, Plan
from .noise import NoiseAugment, NoiseBank, NoiseDraw, draw_noise
from .resample import Resampler
from .s3prl_fbank import S3prlFBank
from .sharding import allreduce_stats, finalize_stats, lpt_partition
from .specaug import draw_masks

__all__ = ["FrontEnd", "Plan", "DeviceCollate", "collate_host_part", "Resampler", "S3prlFBank", "draw_masks", "NoiseBank", "NoiseAugment", "NoiseDraw", "draw_noise", "lpt_partition", "allreduce_stats", "finalize_stats",
           "load_library", "LidfeError", "LIB_PATH", "tables"]
