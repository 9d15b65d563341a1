"""Batched, on-device front-end: packed waveforms -> (B, T_max, n_out) features + wav_percents.

This is the host side of the drop-in: it keeps the feature contract of
``MergedDataset.collate_fn`` (ref: lid/raw_datasets.py:345-365 -- zero padded ``(B, T_max, n_mels)``
batch plus ``wav_percents = T_i / T_max``) and of ``wav2mel(use_kaildi=True)``
(ref: lid/audio_processor.py:41-69), and calls the sm_100a kernels through the C ABI in
``include/lidfe.h``.  PyTorch is only used for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple, Union

import torch

from . import _lib, tables
from .noise import NoiseAugment, NoiseBank, NoiseDraw, noise_table

CMVN_MODES = {"none": _lib.CMVN_NONE, "utt": _lib.CMVN_PER_UTT, "global_apply": _lib.CMVN_APPLY_GLOBAL,
              "global_accum": _lib.CMVN_ACCUM_GLOBAL, "topdb": _lib.POST_TOPDB}
LOG_FLOOR = float(torch.finfo(torch.float32).eps)   # ta: compliance/kaldi.py:22


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _ll_array(values: Sequence[int]):
    return (C.c_longlong * len(values))(*[int(v) for v in values])


@dataclass
class _Layout:
    """What ``FrontEnd.pack`` needs of a plan: where every utterance goes in the packed buffer."""
    lengths: List[int]
    offsets: List[int]
    total_samples: int


@dataclass
class Plan:
    """Segment-offset table of one batch (host copy + the device-side tile table inside ``handle``)."""
    handle: int
    lengths: List[int]          # samples per utterance
    offsets: List[int]          # first sample of each utterance inside the packed buffer
    frames: List[int]           # frames per utterance (kaldi snip_edges)
    out_rows: List[int]         # output row of frame 0 of each utterance
    rows: int                   # rows of the output matrix
    t_max: int                  # longest utterance in frames
    padded: bool                # (B, T_max, n_out) layout if True, packed (sum T_i, n_out) otherwise
    total_samples: int          # length of the packed buffer (including alignment gaps)
    _owner: "FrontEnd" = None

    @property
    def batch(self) -> int:
        return len(self.lengths)

    @property
    def total_frames(self) -> int:
        return sum(self.frames)

    @property
    def wav_percents(self) -> torch.Tensor:
        """T_i / T_max as float32 -- ref: lid/raw_datasets.py:353-354"""
        return torch.tensor([f / self.t_max for f in self.frames], dtype=torch.float32)

    def close(self) -> None:
        if self.handle:
            _lib.load_library().lidfe_plan_destroy(self.handle)
            self.handle = 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FrontEnd:
    """Kaldi-compatible fbank / MFCC + SpecAugment + CMVN on one B200.

    Parameters mirror the ones ``MergedDataset`` forwards to ``wav2mel``
    (ref: lid/raw_datasets.py:196-210,282-291): ``win_length`` / ``hop_length`` in seconds, ``n_mels``,
    ``sr``.  ``preemph`` is the per-frame Kaldi coefficient (1.0 in the reference's call,
    ref: lid/audio_processor.py:60).  ``n_ceps > 0`` selects the MFCC epilogue
    (ta: compliance/kaldi.py:669-813; the reference itself has no MFCC).
    """

    def __init__(self, n_mels: int = 80, n_ceps: int = 0, sr: int = 16000, win_length: float = 0.025,
                 hop_length: float = 0.01, preemph: float = 1.0, cepstral_lifter: float = 22.0,
                 remove_dc: bool = True, in_dtype: torch.dtype = torch.float32, in_scale: float = 1.0,
                 device: Union[str, torch.device, None] = None, kind: str = "kaldi", pad: int = 0,
                 top_db: float = 80.0, window: str = "povey", dither: float = 0.0, seed: int = 0,
                 precise: bool = False):
        """``kind="kaldi"``: the ``use_kaildi=True`` branch (ref: lid/audio_processor.py:41-69).
        ``kind="melspec_db"``: the reference's default branch, MelSpectrogram(n_fft=512, win 400, hop 160, pad,
        center, reflect, power 2, HTK mel 0-8 kHz) + AmplitudeToDB(top_db=80) (ref: lid/audio_processor.py:72-105);
        ``preemph`` / ``remove_dc`` / ``n_ceps`` do not apply to it.
        ``window``: one of torchaudio.compliance.kaldi's window types -- "povey" (the reference's), "hanning", "hamming",
        "rectangular", "blackman" (ta: compliance/kaldi.py:86-113); kaldi branch only.
        ``dither`` > 0: ``wav += dither * U[0,1)`` (ref: lid/audio_processor.py:129) inside the fused kernel, Philox keyed
        by (seed, utterance, sample); 0 is the reference's ``wav2mel`` (its kaldi call passes dither=0.0, :57).
        ``precise=True`` (either kind; not with in-kernel dither): the same formula evaluated in float64 on the same fp32 tables and rounded once
        (``lidfe_set_precision``): at least as close to the fp64 truth as the reference's own fp32 result on every mel
        bin, at about 3 x the time of the default fast fp32 kernels."""
        if kind not in ("kaldi", "melspec_db"):
            raise ValueError("kind must be 'kaldi' or 'melspec_db'")
        self.kind = kind
        if kind == "melspec_db":
            preemph, remove_dc, n_ceps = 0.0, False, 0
            if window != "povey" or dither != 0.0:
                raise ValueError("window / dither belong to kind='kaldi'")
        wtypes = {"povey": _lib.WINDOW_POVEY, "hanning": _lib.WINDOW_HANNING, "hamming": _lib.WINDOW_HAMMING,
                  "rectangular": _lib.WINDOW_RECTANGULAR, "blackman": _lib.WINDOW_BLACKMAN}
        if window not in wtypes:
            raise ValueError("Invalid window type " + str(window))      # ta: compliance/kaldi.py:113
        self.lib = _lib.load_library()
        if not torch.cuda.is_available():
            raise RuntimeError("speech_lid_b200.FrontEnd needs a CUDA device (sm_100a); there is no CPU path")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        if in_dtype not in (torch.float32, torch.int16):
            raise ValueError("in_dtype must be torch.float32 or torch.int16")
        # seconds -> milliseconds -> samples exactly as the reference + torchaudio do
        # (ref: lid/audio_processor.py:50-51; ta: compliance/kaldi.py:138-140)
        if kind == "melspec_db":       # samples straight from seconds (ref: lid/audio_processor.py:89-90)
            frame_len = int(sr * win_length)
            frame_shift = int(sr * hop_length)
        else:
            frame_len = int(sr * int(1000 * win_length) * 0.001)
            frame_shift = int(sr * int(1000 * hop_length) * 0.001)
        fft_len = 1 if frame_len == 0 else 2 ** (frame_len - 1).bit_length()
        self.cfg = _lib.LidfeConfig(sample_rate=int(sr), frame_len=frame_len, frame_shift=frame_shift,
                                    fft_len=fft_len, n_mels=int(n_mels), n_ceps=int(n_ceps),
                                    preemph=float(preemph), remove_dc=int(bool(remove_dc)),
                                    log_floor=LOG_FLOOR if kind == "kaldi" else 1e-10,
                                    in_dtype=_lib.IN_I16 if in_dtype == torch.int16 else _lib.IN_F32,
                                    in_scale=float(in_scale),
                                    framing=_lib.FRAMING_KALDI if kind == "kaldi" else _lib.FRAMING_CENTER,
                                    pad=int(pad) if kind == "melspec_db" else 0,
                                    log_kind=_lib.LOG_NATURAL if kind == "kaldi" else _lib.LOG_DB10,
                                    top_db=float(top_db), dither=float(dither),
                                    window_type=wtypes[window] if kind == "kaldi" else _lib.WINDOW_HANN_PERIODIC,
                                    seed=int(seed) & 0xFFFFFFFFFFFFFFFF)
        self.in_dtype = in_dtype
        self.n_mels, self.n_ceps = int(n_mels), int(n_ceps)
        self.n_out = self.n_ceps if self.n_ceps > 0 else self.n_mels
        self.frame_len, self.frame_shift = frame_len, frame_shift
        self.align = 8 if in_dtype == torch.int16 else 4     # samples per 16 bytes (TMA bulk copy granularity)
        if frame_len != 400 or frame_shift != 160 or int(sr) != 16000:
            _lib.check(_lib.E_CONFIG)
        if kind == "kaldi":
            window = tables.kaldi_window(window, frame_len).contiguous()
            banks = tables.mel_banks(self.n_mels, fft_len, float(sr)).contiguous()
        else:
            window = tables.hann_window(frame_len).contiguous()
            banks = tables.htk_mel_banks(self.n_mels, fft_len).contiguous()
        dct = tables.dct_matrix(self.n_ceps, self.n_mels).contiguous() if self.n_ceps > 0 else None
        lift = tables.lifter(self.n_ceps, cepstral_lifter).contiguous() if self.n_ceps > 0 else None
        self._tables = (window, banks, dct, lift)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lidfe_create(C.byref(h), C.byref(self.cfg), _ptr(window), _ptr(banks), _ptr(dct),
                                             _ptr(lift)))
        self.handle = h.value
        self.precise = bool(precise)
        if self.precise:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.lidfe_set_precision(self.handle, 1))

    def close(self) -> None:
        if getattr(self, "handle", None):
            for cache in (self.__dict__.get("_plan_cache", {}), ):
                for plan in list(cache.values()):
                    plan.close()
                cache.clear()
            for st in self.__dict__.get("_host_cache", {}).values():
                for c in st:
                    c["plan"].close()
            self.__dict__.get("_host_cache", {}).clear()
            self.lib.lidfe_destroy(self.handle)      # plans still alive elsewhere keep the native handle until they go
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ measurement hooks
    def profile_begin(self, max_launches: int, stride: int = 1) -> None:
        """Bracket the fused fbank kernel of every ``stride``-th featurize call with a CUDA event pair."""
        _lib.check(self.lib.lidfe_profile_set_stride(self.handle, int(stride)))
        _lib.check(self.lib.lidfe_profile_begin(self.handle, int(max_launches)))

    def profile_end(self) -> List[float]:
        """Per-launch durations (ms) of the fused fbank kernel since profile_begin()."""
        cap = 1 << 16
        buf = (C.c_float * cap)()
        n = C.c_int(0)
        _lib.check(self.lib.lidfe_profile_end(self.handle, buf, cap, C.byref(n)))
        return [float(buf[i]) for i in range(min(n.value, cap))]

    def pool_stats(self) -> Tuple[int, int]:
        """(plan-memory blocks allocated since creation, blocks currently free in the pool)."""
        a, f = C.c_longlong(0), C.c_longlong(0)
        _lib.check(self.lib.lidfe_pool_stats(self.handle, C.byref(a), C.byref(f)))
        return int(a.value), int(f.value)

    # ------------------------------------------------------------------ frame arithmetic
    def num_frames(self, n_samples: int) -> int:
        """kaldi: 1 + (N - 400) // 160 (0 if N < 400), ta: compliance/kaldi.py:63-67;
        melspec_db: 1 + (N + 2 pad) // 160 (torch.stft, center=True)"""
        return int(self.lib.lidfe_num_frames(int(n_samples), C.byref(self.cfg)))

    # ------------------------------------------------------------------ planning / packing
    def make_plan(self, lengths: Sequence[int], padded: bool = True,
                  offsets: Optional[Sequence[int]] = None, t_max: Optional[int] = None,
                  stream: Optional[torch.cuda.Stream] = None) -> Plan:
        """Build the segment-offset table for utterances of ``lengths`` samples.  ``offsets`` default to a
        packing that starts every utterance on a 16-byte boundary (so each tile is one TMA bulk copy)."""
        lengths = [int(n) for n in lengths]
        if offsets is None:
            offsets, pos = [], 0
            for n in lengths:
                offsets.append(pos)
                pos += (n + self.align - 1) // self.align * self.align
            total = pos
        else:
            offsets = [int(o) for o in offsets]
            total = max(o + n for o, n in zip(offsets, lengths)) if lengths else 0
        frames = [self.num_frames(n) for n in lengths]
        for n, f in zip(lengths, frames):
            if f <= 0:
                _lib.check(_lib.E_SHORT)
        if t_max is None:
            t_max = max(frames)
        elif t_max < max(frames):
            raise ValueError("t_max smaller than the longest utterance")
        if padded:
            out_rows = [i * t_max for i in range(len(lengths))]
            rows = len(lengths) * t_max
            pad_rows = _ll_array([t_max] * len(lengths))
        else:
            out_rows, acc = [], 0
            for f in frames:
                out_rows.append(acc)
                acc += f
            rows = acc
            pad_rows = None
        ph = C.c_void_p()
        with torch.cuda.device(self.device):
            # one pinned-buffer fill + one async copy on the current stream; the memory comes from the handle's pool, so
            # a new length signature every step costs no cudaMalloc / synchronisation (include/lidfe.h, Conventions)
            st = stream if stream is not None else torch.cuda.current_stream(self.device)
            _lib.check(self.lib.lidfe_plan_create_async(self.handle, C.byref(ph), len(lengths), _ll_array(offsets),
                                                        _ll_array(lengths), _ll_array(out_rows), pad_rows,
                                                        st.cuda_stream))
        return Plan(handle=ph.value, lengths=lengths, offsets=offsets, frames=frames, out_rows=out_rows,
                    rows=rows, t_max=t_max, padded=padded, total_samples=total, _owner=self)

    def cached_plan(self, lengths: Sequence[int], padded: bool = True) -> Plan:
        """``make_plan`` behind a small LRU keyed by the batch's length signature: repeated shapes (fixed-length
        batches, the single-utterance wrappers) skip the table upload.  A plan owns device workspace, so one plan is
        meant to be in flight on one stream at a time."""
        key = (tuple(int(n) for n in lengths), bool(padded))
        cache = self.__dict__.setdefault("_plan_cache", {})
        plan = cache.pop(key, None)
        if plan is None:
            plan = self.make_plan(lengths, padded=padded)
            while len(cache) >= 16:
                cache.pop(next(iter(cache)))
        cache[key] = plan
        return plan

    def pack(self, wavs: Sequence[torch.Tensor], plan: Plan, pinned: Optional[torch.Tensor] = None,
             stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """Copy a list of (N_i,) / (1, N_i) waveforms (host or device) into one packed device buffer laid out
        by ``plan``.  Host inputs go through one pinned staging buffer and one H2D copy."""
        flat = []
        for w in wavs:
            if w.dim() == 2:
                w = w[0]        # channel=-1 -> first channel     ta: compliance/kaldi.py:135-137
            flat.append(w)
        if stream is not None:
            with torch.cuda.stream(stream):
                return self.pack(flat, plan, pinned=pinned)
        if all(w.is_cuda for w in flat):
            packed = torch.zeros(plan.total_samples, dtype=self.in_dtype, device=self.device)
            for w, o, n in zip(flat, plan.offsets, plan.lengths):
                packed[o:o + n].copy_(w.to(self.in_dtype), non_blocking=True)
            return packed
        # host inputs: the native packer (lidfe_pack_host, a few host threads) gathers them into a persistent pinned
        # staging buffer -- two of them alternate, each guarded by the event of its last H2D copy, so nothing is
        # pinned / allocated per batch and the packer of batch i+1 never overwrites bytes batch i is still shipping
        host = []
        for w in flat:
            if w.is_cuda:
                w = w.cpu()
            if w.dtype != self.in_dtype or not w.is_contiguous():
                w = w.to(self.in_dtype).contiguous()
            host.append(w)
        cur = torch.cuda.current_stream(self.device)
        # (is_pinned() is a driver query per tensor: the first and the last item decide -- a DataLoader pins all of a
        # batch or none; a pageable straggler would still be copied correctly by cudaMemcpyAsync, only synchronously)
        if pinned is None and host[0].is_pinned() and host[-1].is_pinned():
            # already pinned (DataLoader(pin_memory=True)): no staging copy, one async copy per utterance straight to its
            # place; the sources are kept referenced until the stream has passed the copies
            keep = self.__dict__.setdefault("_h2d_keep", [])
            while keep and keep[0][0].query():
                keep.pop(0)
            with torch.cuda.device(self.device):
                dev = torch.zeros(plan.total_samples, dtype=self.in_dtype, device=self.device)
                ptrs = (C.c_void_p * len(host))(*[w.data_ptr() for w in host])
                _lib.check(self.lib.lidfe_h2d_gather(dev.data_ptr(), ptrs, _ll_array(plan.offsets), _ll_array(plan.lengths),
                                                     len(host), dev.element_size(), cur.cuda_stream))
                done = torch.cuda.Event()
                done.record(cur)
            keep.append((done, host))
            return dev
        if pinned is not None and pinned.numel() >= plan.total_samples:
            stage, ev = pinned, None
        else:
            stage, ev = self._staging(plan.total_samples)
        B = len(host)
        total, eb = plan.total_samples, stage.element_size()
        # large batches go in a few groups of utterances: the H2D copy of one group runs while the next one is packed
        groups = max(1, min(B, 4, (total * eb) >> 24))
        bounds = [0]
        for k in range(1, groups):
            target = total * k // groups
            i = bounds[-1]
            while i < B and plan.offsets[i] < target:
                i += 1
            bounds.append(max(i, bounds[-1]))
        bounds.append(B)
        with torch.cuda.device(self.device):
            dev = torch.empty(total, dtype=self.in_dtype, device=self.device)
            for k in range(groups):
                a, b = bounds[k], bounds[k + 1]
                if a == b:
                    continue
                lo = plan.offsets[a]
                hi = plan.offsets[b] if b < B else total
                ptrs = (C.c_void_p * (b - a))(*[w.data_ptr() for w in host[a:b]])
                _lib.check(self.lib.lidfe_pack_host(stage.data_ptr() + lo * eb, ptrs, _ll_array([o - lo for o in plan.offsets[a:b]]),
                                                    _ll_array(plan.lengths[a:b]), b - a, eb, hi - lo, int(self.pack_threads)))
                dev[lo:hi].copy_(stage[lo:hi], non_blocking=True)
            if ev is not None:
                ev.record(cur)
        return dev

    # host threads of the native packer (lidfe_pack_host): up to 16, the host's cores shared between the local ranks
    pack_threads = max(1, min(16, (os.cpu_count() or 8) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))

    def _staging(self, n: int):
        """One of two persistent pinned staging buffers of at least ``n`` elements, free for reuse (its last H2D copy
        has completed), with the event the caller records after shipping it."""
        st = self.__dict__.setdefault("_stage", {"bufs": [None, None], "evs": [None, None], "i": 0})
        i = st["i"] = st["i"] ^ 1
        if st["evs"][i] is None:
            st["evs"][i] = torch.cuda.Event()
        else:
            st["evs"][i].synchronize()
        if st["bufs"][i] is None or st["bufs"][i].numel() < n:
            st["bufs"][i] = torch.empty(int(n * 1.25) + 1024, dtype=self.in_dtype).pin_memory()
        return st["bufs"][i], st["evs"][i]

    # ------------------------------------------------------------------ the hot path
    def featurize_packed(self, packed: torch.Tensor, plan: Plan, out: Optional[torch.Tensor] = None,
                         masks: Optional[torch.Tensor] = None, cmvn: str = "none",
                         stats_in: Optional[torch.Tensor] = None, stats_out: Optional[torch.Tensor] = None,
                         stream: Optional[torch.cuda.Stream] = None, raw: bool = False) -> torch.Tensor:
        """Launch the fused kernel on device-resident packed samples.  Returns ``out``:
        (B, T_max, n_out) if the plan is padded, (sum T_i, n_out) otherwise.
        ``raw=True``: ``packed`` holds raw samples (int16 PCM scaled by ``in_scale``, or float32) and
        ``read_audio``'s ``normalize_wav`` (ref: lid/audio_processor.py:108-122) is fused in: a statistics pre-pass, then
        (x - mean) / (std + 1e-6) applied while the kernel stages each tile."""
        if self.kind == "melspec_db":
            # the reference's default branch always ends in AmplitudeToDB(top_db=80); it has no CMVN
            if cmvn not in ("none", "topdb"):
                raise ValueError("kind='melspec_db' supports no CMVN (ref: lid/audio_processor.py:72-105)")
            cmvn = "topdb"
        elif cmvn == "topdb":
            raise ValueError("cmvn='topdb' belongs to kind='melspec_db'")
        if raw and getattr(self, "precise", False):
            raise ValueError("precise=True does not serve the fused normalize_wav load (raw=True): normalise with "
                             "wave_stages first, or use the default arithmetic")
        if packed.dtype != self.in_dtype or not packed.is_cuda or not packed.is_contiguous():
            raise ValueError("packed must be a contiguous CUDA tensor of dtype %s" % self.in_dtype)
        if packed.numel() < plan.total_samples:
            raise ValueError("packed buffer shorter than the plan's extent")
        if out is None:
            shape = (plan.batch, plan.t_max, self.n_out) if plan.padded else (plan.rows, self.n_out)
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        if out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous() or out.numel() < plan.rows * self.n_out:
            raise ValueError("out must be a contiguous float32 CUDA tensor with rows*n_out elements")
        n_masks = 0
        if masks is not None:
            if masks.dtype != torch.int32 or masks.dim() != 3 or masks.shape[0] != plan.batch or masks.shape[2] != 4:
                raise ValueError("masks must be int32 [B, n_masks, 4]")
            if not masks.is_cuda:
                # pinned + non-blocking: a pageable copy would hold the host until everything queued ahead of it on the
                # stream (the waveforms' H2D copies) has drained
                masks = masks.contiguous().pin_memory().to(self.device, non_blocking=True)
            masks = masks.to(self.device).contiguous()
            n_masks = masks.shape[1]
            if n_masks == 0:
                masks = None
        for s in (stats_in, stats_out):
            if s is not None and (s.dtype != torch.float64 or s.numel() != 2 * self.n_out + 1 or not s.is_cuda):
                raise ValueError("stats tensors must be float64 CUDA tensors of 2*n_out+1 elements")
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        fn = self.lib.lidfe_featurize_raw if raw else self.lib.lidfe_featurize
        with torch.cuda.device(self.device):
            _lib.check(fn(self.handle, plan.handle, packed.data_ptr(), out.data_ptr(), self.n_out, _ptr(masks), n_masks,
                          CMVN_MODES[cmvn], _ptr(stats_in), _ptr(stats_out), st.cuda_stream))
        return out

    # ------------------------------------------------------------------ argument checks shared by the entry points
    def _check_feats(self, feats: torch.Tensor, plan: Plan) -> None:
        if (feats.dtype != torch.float32 or not feats.is_cuda or not feats.is_contiguous()
                or feats.numel() < plan.rows * self.n_out or feats.device != self.device):
            raise ValueError("feats must be a contiguous float32 tensor on %s with rows*n_out elements" % self.device)

    def _check_masks(self, masks: Optional[torch.Tensor], plan: Plan):
        if masks is None:
            return None, 0
        if masks.dtype != torch.int32 or masks.dim() != 3 or masks.shape[0] != plan.batch or masks.shape[2] != 4:
            raise ValueError("masks must be int32 [B, n_masks, 4]")
        if masks.shape[1] == 0:
            return None, 0
        return masks.to(self.device).contiguous(), int(masks.shape[1])

    def _check_stats(self, stats: torch.Tensor) -> None:
        if (stats.dtype != torch.float64 or stats.numel() != 2 * self.n_out + 1 or not stats.is_cuda
                or not stats.is_contiguous() or stats.device != self.device):
            raise ValueError("stats must be a contiguous float64 tensor of 2*n_out+1 elements on %s "
                             "(move the all-reduced vector back to the GPU)" % self.device)

    def cmvn_apply(self, feats: torch.Tensor, plan: Plan, stats: torch.Tensor,
                   masks: Optional[torch.Tensor] = None, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """Second pass of global CMVN, in place: (x - mean) / (std + 1e-9) from the all-reduced sums, then masks."""
        self._check_feats(feats, plan)
        self._check_stats(stats)
        masks, n_masks = self._check_masks(masks, plan)
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lidfe_cmvn_apply(self.handle, plan.handle, feats.data_ptr(), self.n_out, _ptr(masks),
                                                 n_masks, stats.data_ptr(), st.cuda_stream))
        return feats

    def mask_apply(self, feats: torch.Tensor, plan: Plan, masks: torch.Tensor,
                   stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """Zero-fill [t0,t1) x [f0,f1) bands in place (SpecAugment application, ref: lid/audio_processor.py:225-227)."""
        self._check_feats(feats, plan)
        masks, n_masks = self._check_masks(masks, plan)
        if masks is None:
            return feats
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.lidfe_mask_apply(self.handle, plan.handle, feats.data_ptr(), self.n_out,
                                                 masks.data_ptr(), n_masks, st.cuda_stream))
        return feats

    def wave_stages(self, packed: torch.Tensor, plan: Plan, normalize: bool = False, dither: float = 0.0,
                    noise: Optional[torch.Tensor] = None, preemph: float = 0.0,
                    stream: Optional[torch.cuda.Stream] = None, out: Optional[torch.Tensor] = None,
                    pcm_scale: float = 1.0 / 32768.0) -> torch.Tensor:
        """normalize_wav / dither / 0.97 pre-emphasis over every utterance of a packed float32 buffer
        (ref: lid/audio_processor.py:108-115,129-134).  ``dither`` without ``noise``: the U[0,1) draw happens on the
        device (Philox keyed by (seed, utterance, sample)); with ``noise`` (the reference's ``torch.rand_like`` draw) the
        result is bit-identical to the reference.  ``packed`` may be int16 PCM (scaled by ``pcm_scale`` first, as
        torchaudio.load does).  Returns a new packed float32 buffer (or fills ``out``)."""
        if packed.dtype not in (torch.float32, torch.int16):
            raise ValueError("wave_stages works on float32 samples or int16 PCM")
        if not packed.is_cuda or not packed.is_contiguous() or packed.numel() < plan.total_samples:
            raise ValueError("packed must be a contiguous CUDA buffer covering the plan's extent")
        if noise is not None and (noise.dtype != torch.float32 or not noise.is_cuda or not noise.is_contiguous()
                                  or noise.numel() < plan.total_samples):
            raise ValueError("noise must be a contiguous float32 CUDA buffer laid out like `packed`")
        if out is not None and (out.dtype != torch.float32 or not out.is_cuda or out.numel() < plan.total_samples):
            raise ValueError("out must be a float32 CUDA buffer covering the plan's extent")
        if out is None:
            out = torch.zeros(packed.numel(), dtype=torch.float32, device=packed.device)
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            if packed.dtype == torch.int16:
                _lib.check(self.lib.lidfe_wave_stages_i16(self.handle, plan.handle, packed.data_ptr(), float(pcm_scale),
                                                          out.data_ptr(), int(normalize), float(dither), _ptr(noise),
                                                          float(preemph), st.cuda_stream))
            else:
                _lib.check(self.lib.lidfe_wave_stages(self.handle, plan.handle, packed.data_ptr(), out.data_ptr(),
                                                      int(normalize), float(dither), _ptr(noise), float(preemph),
                                                      st.cuda_stream))
        return out

    def add_noise(self, packed: torch.Tensor, plan: Plan, draw: NoiseDraw, bank: Optional[NoiseBank] = None,
                  normalize: bool = False, out: Optional[torch.Tensor] = None,
                  stream: Optional[torch.cuda.Stream] = None, pcm_scale: float = 1.0 / 32768.0) -> torch.Tensor:
        """Additive noise at each utterance's SNR (``torchaudio.functional.add_noise``; ``noise.py``), then
        ``normalize_wav`` when ``normalize``: the evaluation chain "load -> add noise -> read_audio(normalize=True)".
        ``draw`` comes from ``draw_noise`` (with the same ``bank``; ``bank=None`` mixes N(0,1) drawn on the device from
        ``draw.seed``).  ``packed`` is float32 or int16 PCM (scaled by ``pcm_scale`` first).  Returns a new packed
        float32 buffer with zeroed gaps (or fills ``out``).  Unlike torchaudio, a zero-energy noise window leaves the
        utterance clean instead of NaN."""
        if packed.dtype not in (torch.float32, torch.int16):
            raise ValueError("add_noise works on float32 samples or int16 PCM")
        if not packed.is_cuda or not packed.is_contiguous() or packed.numel() < plan.total_samples:
            raise ValueError("packed must be a contiguous CUDA buffer covering the plan's extent")
        if out is not None and (out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous()
                                or out.numel() < plan.total_samples):
            raise ValueError("out must be a contiguous float32 CUDA buffer covering the plan's extent")
        if bank is not None and bank.data.device != packed.device:
            raise ValueError("the noise bank lives on %s, the samples on %s" % (bank.data.device, packed.device))
        tab, snr = noise_table(draw, bank, plan.batch)
        i16 = packed.dtype == torch.int16
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        # the output and the per-utterance tables are allocated and uploaded on the launching stream: nothing is
        # ordered on another stream, so a side-stream caller needs no synchronisation
        with torch.cuda.device(self.device), torch.cuda.stream(st):
            if out is None:
                out = torch.zeros(packed.numel(), dtype=torch.float32, device=packed.device)
            snr_d = snr.pin_memory().to(self.device, non_blocking=True)
            tab_d = tab.pin_memory().to(self.device, non_blocking=True) if tab is not None else None
            _lib.check(self.lib.lidfe_add_noise(self.handle, plan.handle, packed.data_ptr(), int(i16),
                                                float(pcm_scale) if i16 else 1.0, out.data_ptr(),
                                                _ptr(bank.data) if bank is not None else None,
                                                bank.data.numel() if bank is not None else 0, _ptr(tab_d),
                                                snr_d.data_ptr(), int(draw.seed) & 0xFFFFFFFFFFFFFFFF, int(normalize),
                                                st.cuda_stream))
        return out

    def featurize_host(self, host_in: torch.Tensor, plan: Plan, host_out: torch.Tensor,
                       masks: Optional[torch.Tensor] = None, cmvn: str = "none", chunks: int = 8) -> torch.Tensor:
        """Host-buffer entry (what a CPU-side caller of the reference's ``wav2mel`` sees): ``host_in`` is the packed
        waveform buffer laid out by ``plan`` in (ideally pinned) host memory, ``host_out`` receives the padded
        ``(B, T_max, n_out)`` batch.  The batch is cut into ``chunks`` groups of utterances, each on its own stream, so
        the H2D copy of one group, the kernels of the previous one and the D2H copy of the one before overlap
        (PCIe is full duplex).  Returns ``host_out`` after synchronising.

        ``host_in`` may also hold raw int16 PCM (what a 16-bit wav file decodes to): each group is then shipped at
        2 bytes per sample and ``read_audio``'s scaling + ``normalize_wav`` (ref: lid/audio_processor.py:108-122) run on
        the device before framing."""
        pcm = host_in.dtype == torch.int16
        # int16 PCM into an int16 FrontEnd(in_scale=1/32768): ONE fused pass (statistics pre-pass + normalise-at-load);
        # into a float32 FrontEnd: the two-kernel path (wave_stages writes a float32 copy the fbank kernel re-reads)
        fused = pcm and self.in_dtype == torch.int16
        if not plan.padded:
            raise ValueError("featurize_host needs a padded plan")
        if cmvn not in ("none", "utt", "topdb"):
            raise ValueError("featurize_host supports cmvn 'none' or 'utt' (global CMVN needs the all-reduce in between)")
        B = plan.batch
        chunks = max(1, min(chunks, B))
        # the pipeline (sub-plans, device buffers, streams) is keyed by the batch's CONTENT, not by the plan's address:
        # a freed plan's handle is routinely handed out again by the allocator for a different batch
        key = (tuple(plan.lengths), tuple(plan.offsets), plan.t_max, chunks, pcm)
        cache = self.__dict__.setdefault("_host_cache", {})
        st = cache.get(key)
        if st is None:
            bounds = [(B * c) // chunks for c in range(chunks + 1)]
            st = []
            for c in range(chunks):
                a, b = bounds[c], bounds[c + 1]
                base = plan.offsets[a]
                end = plan.offsets[b] if b < B else plan.total_samples
                sub = self.make_plan(plan.lengths[a:b], padded=True, offsets=[o - base for o in plan.offsets[a:b]],
                                     t_max=plan.t_max)
                st.append(dict(a=a, b=b, base=base, end=end, plan=sub, stream=torch.cuda.Stream(self.device),
                               dev_in=torch.empty(end - base, dtype=host_in.dtype, device=self.device),
                               dev_f32=(torch.zeros(end - base, dtype=torch.float32, device=self.device)
                                        if pcm and not fused else None),
                               dev_out=torch.empty((b - a, plan.t_max, self.n_out), dtype=torch.float32, device=self.device)))
            torch.cuda.current_stream(self.device).synchronize()      # sub-plan tables were uploaded on this stream
            cache.clear()          # one cached pipeline at a time
            cache[key] = st
        cur = torch.cuda.current_stream(self.device)
        for c in st:
            s = c["stream"]
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                c["dev_in"].copy_(host_in[c["base"]:c["end"]], non_blocking=True)
                m = None
                if masks is not None and masks.shape[1] > 0:
                    m = masks[c["a"]:c["b"]].to(self.device, non_blocking=True)
                src = c["dev_in"]
                if pcm and not fused:
                    src = self.wave_stages(c["dev_in"], c["plan"], normalize=True, stream=s, out=c["dev_f32"])
                self.featurize_packed(src, c["plan"], out=c["dev_out"], masks=m, cmvn=cmvn, stream=s, raw=fused)
                host_out[c["a"]:c["b"]].copy_(c["dev_out"], non_blocking=True)
        for c in st:
            c["stream"].synchronize()
        return host_out

    def featurize(self, wavs: Sequence[torch.Tensor], masks: Optional[torch.Tensor] = None, cmvn: str = "none",
                  padded: bool = True, cache_plan: bool = True,
                  noise: Optional[NoiseAugment] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """The batched public entry: list of waveforms -> ``(feats, wav_percents)`` with the collate contract
        (ref: lid/raw_datasets.py:345-365).  ``feats`` stays on the device -- that is where the model consumes it.
        ``cache_plan=False`` (ragged training batches: every batch has its own length signature): the plan is built for
        this call and handed straight back to the handle's pool -- the pool re-uses its block only after the work
        launched here has finished (an event per block), so nothing is allocated or freed in steady state.
        ``masks`` may be a callable ``frames -> int32 [B, n_masks, 4]``: it is evaluated after the H2D copies have been
        issued (``DeviceCollate`` draws its SpecAugment bounds this way, under the DMA).
        ``noise``: a ``NoiseAugment``; every call draws its noise and mixes it into the packed waveforms
        (``add_noise``) before the features are computed.  Needs a float32 FrontEnd."""
        if noise is not None and self.in_dtype != torch.float32:
            raise ValueError("noise augmentation needs a float32 FrontEnd (add_noise produces float32 samples)")
        lengths = [int(w.shape[-1]) for w in wavs]
        if cache_plan:
            plan = self.cached_plan(lengths, padded=padded)
            packed = self.pack(wavs, plan)
        else:
            # ship first, plan afterwards: the layout (16-byte aligned prefix sums) is all the packer needs, so the H2D
            # copies are already running while the host fills the plan tables and draws the masks
            if lengths and min(lengths) < self.frame_len:
                _lib.check(_lib.E_SHORT)
            offsets, pos = [], 0
            for n in lengths:
                offsets.append(pos)
                pos += (n + self.align - 1) // self.align * self.align
            packed = self.pack(wavs, _Layout(lengths=lengths, offsets=offsets, total_samples=pos))
            plan = self.make_plan(lengths, padded=padded, offsets=offsets)
        if noise is not None:
            packed = self.add_noise(packed, plan, noise.draw(plan.batch), bank=noise.bank, normalize=noise.normalize)
        if callable(masks):
            masks = masks(plan.frames)
        out = self.featurize_packed(packed, plan, masks=masks, cmvn=cmvn)
        percents = plan.wav_percents
        if not cache_plan:
            plan.close()
        return out, percents
