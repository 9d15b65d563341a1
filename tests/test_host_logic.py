"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol include/lidfe.h declares,
argument validation, frame arithmetic, table construction, mask drawing, sharding.  No compute calls (no GPU here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import speech_lid_b200 as lid
from speech_lid_b200 import _lib, tables
from oracle import frontend_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "lidfe.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(lidfe_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 18
    lib = lid.load_library()
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, "liblidfe.so does not export %s" % missing
    assert sorted(_lib.EXPORTS) == declared, "python binding and header disagree"
    assert lib.lidfe_abi_version() == _lib.ABI_VERSION == 8


def _cfg(**kw):
    base = dict(sample_rate=16000, frame_len=400, frame_shift=160, fft_len=512, n_mels=80, n_ceps=0, preemph=1.0,
                remove_dc=1, log_floor=1.1920929e-07, in_dtype=0, in_scale=1.0)
    base.update(kw)
    return _lib.LidfeConfig(**base)


def test_num_frames_matches_kaldi_snip_edges():
    lib = lid.load_library()
    cfg = _cfg()
    for n in list(range(0, 1300)) + [16000, 48000, 64000, 128000, 320000, 2 ** 31 + 5]:
        assert lib.lidfe_num_frames(n, C.byref(cfg)) == O.kaldi_num_frames(n), n
    assert lib.lidfe_num_frames(1000, None) == 0


def test_error_codes_and_messages():
    lib = lid.load_library()
    assert lib.lidfe_strerror(0) == b"ok"
    for rc in range(-7, 0):
        assert lib.lidfe_strerror(rc).startswith(b"lidfe:")
    with pytest.raises(AssertionError):        # too-short utterance mirrors torchaudio's assertion
        _lib.check(_lib.E_SHORT)
    with pytest.raises(lid.LidfeError) as e:
        _lib.check(_lib.E_CONFIG)
    assert e.value.rc == _lib.E_CONFIG
    _lib.check(0)


def test_create_validates_arguments_before_touching_the_device():
    lib = lid.load_library()
    h = C.c_void_p()
    win = tables.povey_window(400).contiguous()
    banks = tables.mel_banks(80, 512, 16000.0).contiguous()
    assert lib.lidfe_create(None, C.byref(_cfg()), win.data_ptr(), banks.data_ptr(), None, None) == _lib.E_NULL
    assert lib.lidfe_create(C.byref(h), C.byref(_cfg()), None, banks.data_ptr(), None, None) == _lib.E_NULL
    for bad in (dict(sample_rate=8000), dict(frame_len=200), dict(frame_shift=80), dict(fft_len=256),
                dict(n_mels=128), dict(n_mels=2), dict(n_ceps=81), dict(preemph=1.5), dict(in_dtype=7),
                dict(framing=3), dict(pad=16), dict(log_kind=2), dict(log_floor=0.0)):
        assert lib.lidfe_create(C.byref(h), C.byref(_cfg(**bad)), win.data_ptr(), banks.data_ptr(), None, None) \
            == _lib.E_CONFIG, bad
    assert lib.lidfe_create(C.byref(h), C.byref(_cfg(n_ceps=40)), win.data_ptr(), banks.data_ptr(), None, None) \
        == _lib.E_NULL          # MFCC without a DCT table
    assert lib.lidfe_destroy(None) == _lib.E_NULL and lib.lidfe_plan_destroy(None) == _lib.E_NULL
    assert lib.lidfe_featurize(None, None, None, None, 80, None, 0, 0, None, None, None) == _lib.E_NULL
    if not torch.cuda.is_available():
        # a valid configuration needs the device: the call must fail loudly (cudaError), never fall back
        rc = lib.lidfe_create(C.byref(h), C.byref(_cfg()), win.data_ptr(), banks.data_ptr(), None, None)
        assert rc > 0 and not h.value
        with pytest.raises(RuntimeError):
            lid.FrontEnd()


def test_tables_bit_identical_to_oracle():
    assert torch.equal(tables.povey_window(400), O.povey_window(400))
    for n in (80, 40, 23):
        assert torch.equal(tables.mel_banks(n, 512, 16000.0), O.kaldi_mel_banks(n, 512, 16000.0))
    assert torch.equal(tables.dct_matrix(40, 80), O.kaldi_dct_matrix(40, 80))
    assert torch.equal(tables.dct_matrix(13, 23), O.kaldi_dct_matrix(13, 23))
    assert torch.equal(tables.lifter(40, 22.0), O.kaldi_lifter(40, 22.0).float())
    K = pytest.importorskip("torchaudio.compliance.kaldi")
    ref = torch.nn.functional.pad(K.get_mel_banks(80, 512, 16000.0, 20.0, 0.0, 100.0, -500.0, 1.0)[0], (0, 1))
    assert torch.equal(tables.mel_banks(80, 512, 16000.0), ref)
    assert torch.equal(tables.povey_window(400),
                       K._feature_window_function("povey", 400, 0.42, torch.device("cpu"), torch.float32))


def test_melspec_tables_and_centered_frame_count():
    assert torch.equal(tables.hann_window(400), torch.hann_window(400))
    assert torch.equal(tables.htk_mel_banks(80, 512), O.htk_mel_fbanks(257, 0.0, 8000.0, 80, 16000).t())
    F = pytest.importorskip("torchaudio.functional")
    assert torch.equal(tables.htk_mel_banks(80, 512), F.melscale_fbanks(257, 0.0, 8000.0, 80, 16000).t())
    lib = lid.load_library()
    for pad in (0, 16):
        cfg = _cfg(framing=_lib.FRAMING_CENTER, pad=pad, log_kind=_lib.LOG_DB10, preemph=0.0, remove_dc=0,
                   log_floor=1e-10, top_db=80.0)
        for n in (257, 300, 700, 4000, 16000, 128000):
            assert lib.lidfe_num_frames(n, C.byref(cfg)) == O.num_frames_centered(n, pad=pad)
        assert lib.lidfe_num_frames(256 - 2 * pad, C.byref(cfg)) == 0     # torch.stft refuses to reflect-pad this
    # the HTK bank goes through the same sparsifier / tap placement
    k0, cnt, st = (C.c_int * 80)(), (C.c_int * 80)(), (C.c_int * 80)()
    bt = (C.c_int * 5)()
    assert lib.lidfe_mel_plan(80, tables.htk_mel_banks(80, 512).data_ptr(), k0, cnt, st, bt) == 0
    assert all(b > 0 for b in bt)


def test_mel_plan_is_sparse_exact_and_bank_conflict_free():
    lib = lid.load_library()
    cases = [(n, tables.mel_banks(n, 512, 16000.0).contiguous()) for n in (80, 64, 40, 23)]
    cases += [(n, tables.htk_mel_banks(n, 512).contiguous()) for n in (80, 64)]
    for ci, (n, banks) in enumerate(cases):
        first, cnt, st = (C.c_int * 80)(), (C.c_int * 80)(), (C.c_int * 80)()
        bt = (C.c_int * 5)()
        assert lib.lidfe_mel_plan(n, banks.data_ptr(), first, cnt, st, bt) == 0
        steps = list(bt)
        nz = banks != 0
        # every bin feeds at most two adjacent filters; slot m's run = the bins shared by filters m and m+1
        # (slot 0 also takes the bins below the first centre), each non-zero bin in exactly one run
        owner = {}
        for m in range(n):
            band = m // 16
            assert st[m] <= first[m] or cnt[m] == 0
            assert cnt[m] == 0 or st[m] + steps[band] >= first[m] + cnt[m]
            for k in range(first[m], first[m] + cnt[m]):
                assert k not in owner
                owner[k] = m
                fs = nz[:, k].nonzero().flatten().tolist()
                assert set(fs) <= {m, m + 1}, (m, k, fs)
        assert sorted(owner) == nz.any(0).nonzero().flatten().tolist()
        # 16 lanes of a band: distinct addresses fall into distinct 8-byte bank pairs at every step
        for band in range(5):
            ms = list(range(16 * band, min(n, 16 * band + 16)))
            for i in range(steps[band]):
                by_bank = {}
                for m in ms:
                    by_bank.setdefault((st[m] + i) % 16, set()).add(st[m] + i)
                assert all(len(v) == 1 for v in by_bank.values()), "bank conflict in band %d" % band
        # replaying the plan gives back the dense bank bit for bit
        dense = torch.full((n, 257), 7.0)
        assert lib.lidfe_mel_plan_expand(n, banks.data_ptr(), dense.data_ptr()) == 0
        assert torch.equal(dense, banks)
        if ci == 0:
            assert int(nz.sum()) == 501 and steps == [2, 2, 4, 6, 9]      # the fully-unrolled kernel variant
            assert sum(cnt[m] for m in range(n)) == 255                   # bins 1..255, each read once
    banks = cases[0][1]
    first, cnt, st = (C.c_int * 80)(), (C.c_int * 80)(), (C.c_int * 80)()
    bt = (C.c_int * 5)()
    assert lib.lidfe_mel_plan(80, None, first, cnt, st, bt) == _lib.E_NULL
    assert lib.lidfe_mel_plan(200, banks.data_ptr(), first, cnt, st, bt) == _lib.E_CONFIG
    empty = torch.zeros(80, 257)
    assert lib.lidfe_mel_plan(80, empty.data_ptr(), first, cnt, st, bt) == _lib.E_MELBANK
    dense3 = banks.clone()
    dense3[10, 200] = 0.5                                             # a filter reaching far outside its neighbours
    assert lib.lidfe_mel_plan(80, dense3.data_ptr(), first, cnt, st, bt) == _lib.E_MELBANK


def test_draw_masks_consumes_rng_like_the_reference(golden_dir):
    torch.manual_seed(123)
    table = lid.draw_masks([798], 80, 0.05, 27, 2)
    assert table.dtype == torch.int32 and table.shape == (1, 2, 4)
    assert table[0].tolist() == [[406, 417, 50, 56], [688, 690, 7, 10]]      # SURVEY.md appendix A.2
    # batch order, ragged, including T < 20 (no time mask, no RNG draw)
    frames = [798, 18, 298, 5]
    torch.manual_seed(7)
    a = lid.draw_masks(frames, 80, 0.05, 27, 2)
    torch.manual_seed(7)
    b = [O.draw_mask_bounds(T, 80, 0.05, 27, 2) for T in frames]
    assert a.tolist() == [[list(m) for m in u] for u in b]
    assert a[1, :, :2].abs().sum() == 0 and a[3, :, :2].abs().sum() == 0
    # against the reference's own output
    z = np.load(os.path.join(golden_dir, "specaug.npz"))
    for name in ("t798_default", "t298_yaml", "t18_no_tmask"):
        spec = torch.from_numpy(z["spec_" + name])
        t_mask, f_mask, times, seed = z["kw_" + name]
        torch.manual_seed(int(seed))
        m = lid.draw_masks([spec.shape[2]], 80, float(t_mask), int(f_mask), int(times))
        out = O.apply_mask_bounds(spec, [tuple(int(v) for v in row) for row in m[0]])
        assert torch.equal(out, torch.from_numpy(z["out_" + name])), name
    g = torch.Generator().manual_seed(1)
    assert lid.draw_masks([100], 80, 0.05, 27, 0, generator=g).shape == (1, 0, 4)


def test_lpt_partition():
    g = torch.Generator().manual_seed(3)
    lengths = torch.randint(16000, 320001, (1000,), generator=g).tolist()
    for world in (1, 2, 4, 8):
        shards = lid.lpt_partition(lengths, world)
        assert sorted(i for s in shards for i in s) == list(range(1000))
        loads = [sum(lengths[i] for i in s) for s in shards]
        assert max(loads) - min(loads) <= max(lengths)
        assert shards == lid.lpt_partition(lengths, world)          # deterministic: every rank computes the same split
    assert lid.lpt_partition([5, 5], 4) == [[0], [1], [], []]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "speech-lid_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "frontend_oracle" not in src, f


def test_audio_processor_surface_matches_reference_signatures():
    import inspect
    from speech_lid_b200 import audio_processor as ap
    sig = inspect.signature(ap.wav2mel)
    assert list(sig.parameters) == ["x", "use_kaildi", "win_length", "hop_length", "n_mels", "n_fft", "pad", "sr"]
    assert [p.default for p in sig.parameters.values()][1:] == [False, 0.025, 0.01, 80, 512, 0, 16000]
    sig = inspect.signature(ap.spectrogram_augment)
    assert list(sig.parameters) == ["spec", "sr", "n_mels", "hop_length", "t_mask", "f_mask", "mask_times", "t_stretch"]
    assert [p.default for p in sig.parameters.values()][1:] == [16000, 80, 0.01, 0.05, 27, 0, False]
    assert list(inspect.signature(ap.wav_augment).parameters) == ["wav", "sr", "speed_shift", "pitch_shift", "reverb"]
    assert list(inspect.signature(ap.normalize_wav).parameters) == ["wav"]
    assert list(inspect.signature(ap.read_audio).parameters) == ["audio_path", "normalize"]
    spec = torch.zeros(1, 80, 50)
    assert ap.spectrogram_augment(spec, mask_times=0) is spec           # no masks -> returns its input, like the reference
    with pytest.raises(NotImplementedError):
        ap.spectrogram_augment(spec, mask_times=1, t_stretch=True)
    with pytest.raises(NotImplementedError):
        ap.wav2mel(torch.zeros(1, 16000), n_fft=400)


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """include/lidfe.h compiles as C99 with no torch / CUDA headers in sight, and a C program linked against
    liblidfe.so can call the host-only entry points (what a cgo / JNI / ctypes binding relies on)."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lid.load_library()                                        # raises if the library is not built
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "speech-lid_b200")
    src = tmp_path / "use_lidfe.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "lidfe.h"
int main(void) {
  lidfe_config cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.sample_rate = 16000; cfg.frame_len = 400; cfg.frame_shift = 160; cfg.fft_len = 512; cfg.n_mels = 80;
  if (lidfe_num_frames(128000, &cfg) != 798) return 1;
  if (lidfe_num_frames(399, &cfg) != 0) return 2;
  if (lidfe_abi_version() != LIDFE_ABI_VERSION) return 3;
  if (strstr(lidfe_strerror(LIDFE_E_SHORT), "shorter than one frame") == NULL) return 4;
  if (lidfe_create(NULL, &cfg, NULL, NULL, NULL, NULL) != LIDFE_E_NULL) return 5;
  printf("ok %d\n", lidfe_abi_version());
  return 0;
}
''')
    exe = tmp_path / "use_lidfe"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(root, "include"), str(src),
                    "-o", str(exe), "-L", libdir, "-llidfe", "-Wl,-rpath," + libdir], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    assert out.startswith("ok ")


def test_graft_entry_build_passes():
    """build() is what the driver calls: it must compile (or find the library fresh), import the package and pass its
    own export / ABI-version checks."""
    import __graft_entry__ as g
    g.build()


def test_collate_host_part_matches_reference_semantics():
    """texts / text_percents / paths / langs exactly as MergedDataset.collate_fn builds them
    (ref: lid/raw_datasets.py:353-365), restated inline."""
    g = torch.Generator().manual_seed(3)
    lang2index = {"Persian": 0, "Swahili": 1, "Vietnamese": 2}
    batch = []
    for i, (n, L, lang) in enumerate(((16000, 7, "Swahili"), (9000, 12, "Persian"), (12345, 1, "Vietnamese"))):
        batch.append((torch.randn(1, n, generator=g), torch.randint(1, 40, (L,), generator=g), "utt%d.wav" % i, lang))
    texts, text_percents, paths, langs = lid.collate_host_part(batch, lang2index)
    want_texts = torch.nn.utils.rnn.pad_sequence([b[1] for b in batch]).transpose(1, 0)
    assert torch.equal(texts, want_texts) and texts.shape == (3, 12) and texts.dtype == torch.int64
    assert torch.equal(text_percents, torch.FloatTensor([b[1].shape[-1] / (want_texts.shape[1] + 1e-9) for b in batch]))
    assert paths == ["utt0.wav", "utt1.wav", "utt2.wav"]
    assert torch.equal(langs, torch.LongTensor([1, 0, 2])) and langs.dtype == torch.int64


def test_resample_tables_bit_identical_to_torchaudio():
    import math
    import torchaudio.functional.functional as TF
    for orig in (44100, 22050, 48000, 8000, 11025):
        k, w = tables.sinc_resample_kernel(orig, 16000)
        kr, wr = TF._get_sinc_resample_kernel(orig, 16000, math.gcd(orig, 16000))
        assert w == wr and torch.equal(k, kr[:, 0, :])
        ko, wo, _, _ = O.sinc_resample_kernel(orig, 16000)
        assert wo == w and torch.equal(ko[:, 0, :], k)


def test_draw_masks_vectorised_equals_the_serial_draw():
    """draw_masks draws all uniforms with one torch.rand(K); the definition is mask_along_axis' two torch.rand(1) per
    mask (ta: functional/functional.py:885-958).  Same integers and the same generator state afterwards."""
    import random
    from speech_lid_b200.specaug import draw_masks, _draw_masks_serial
    rnd = random.Random(5)
    for trial in range(120):
        B = rnd.randint(1, 48)
        frames = [rnd.choice([1, 5, 19, 20, 21, 98, 500, 1998, rnd.randint(1, 3000)]) for _ in range(B)]
        t_mask = rnd.choice([0.05, 0.0, 0.1, 0.2])
        n_mels = rnd.choice([80, 40, 23])
        f_mask = rnd.choice([f for f in (27, 0, 1, 15, 80) if f <= n_mels])
        times = rnd.choice([0, 1, 2, 3])
        torch.manual_seed(trial)
        want = _draw_masks_serial(frames, n_mels, t_mask, f_mask, times)
        after_want = torch.rand(1)
        torch.manual_seed(trial)
        got = draw_masks(frames, n_mels, t_mask, f_mask, times)
        after_got = torch.rand(1)
        assert torch.equal(want, got) and torch.equal(after_want, after_got), (trial, frames, t_mask, f_mask, times)


def test_pack_host_gathers_and_zeroes_gaps():
    """lidfe_pack_host (the host half of the collate, ref: lid/raw_datasets.py:345-351): every thread count gives the
    same bytes as a plain per-utterance copy, gaps and tail zeroed, bad arguments rejected."""
    lib = lid.load_library()
    g = torch.Generator().manual_seed(11)
    ll = lambda v: (C.c_longlong * len(v))(*v)
    for dtype, eb in ((torch.float32, 4), (torch.int16, 2)):
        lens = torch.randint(400, 300000, (37,), generator=g).tolist() + [400, 401, 0]
        ws = [(torch.randn(n, generator=g) * 1000).to(dtype) for n in lens]
        offs, pos = [], 0
        for n in lens:
            offs.append(pos)
            pos += (n + 7) // 8 * 8
        total = pos + 333
        want = torch.zeros(total, dtype=dtype)
        for w, o, n in zip(ws, offs, lens):
            want[o:o + n] = w
        ptrs = (C.c_void_p * len(ws))(*[w.data_ptr() for w in ws])
        for threads in (1, 2, 3, 8, 32, 0):
            dst = torch.full((total,), 7, dtype=dtype)
            assert lib.lidfe_pack_host(dst.data_ptr(), ptrs, ll(offs), ll(lens), len(ws), eb, total, threads) == 0
            assert torch.equal(dst, want), (dtype, threads)
        dst = torch.zeros(total, dtype=dtype)
        assert lib.lidfe_pack_host(dst.data_ptr(), ptrs, ll(offs), ll(lens), len(ws), 3, total, 1) == _lib.E_ARG
        assert lib.lidfe_pack_host(dst.data_ptr(), ptrs, ll(offs[::-1]), ll(lens), len(ws), eb, total, 1) == _lib.E_OFFSETS
        assert lib.lidfe_pack_host(dst.data_ptr(), ptrs, ll(offs), ll(lens), len(ws), eb, pos - 1000, 1) == _lib.E_OFFSETS
        assert lib.lidfe_pack_host(None, ptrs, ll(offs), ll(lens), len(ws), eb, total, 1) == _lib.E_NULL


def test_bench_dump_outputs_sample_and_files(tmp_path):
    """bench.py --dump-outputs: the same utterances every run (two builds are compared on them), float32 .npy files
    named after the arrays, under 64 MB for the whole dump; bad arguments are refused before any device work."""
    import subprocess
    import sys
    import bench
    pick = bench.dump_pick()
    assert torch.equal(pick, bench.dump_pick())
    assert pick.numel() == bench.DUMP_UTTS == 128 and torch.equal(pick, pick.unique())
    assert 0 <= int(pick[0]) and int(pick[-1]) < bench.B_UTTS
    assert pick[:8].tolist() == [0, 1, 2, 3, 5, 7, 8, 10] and int(pick.sum()) == 15379
    frames = 1 + (bench.N_SAMPLES - 400) // 160
    assert bench.DUMP_UTTS * frames * bench.N_MELS * 4 <= 64 * 10 ** 6
    feats = torch.randn(bench.B_UTTS, 7, bench.N_MELS).index_select(0, pick)
    bench.write_outputs(str(tmp_path / "d"), {"features": feats})
    got = np.load(str(tmp_path / "d" / "features.npy"))
    assert got.dtype == np.float32 and got.shape == (128, 7, bench.N_MELS)
    assert np.array_equal(got, feats.numpy())
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "r")]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + bad, capture_output=True, text=True)
        assert r.returncode == 2 and "error" in r.stderr, bad
    assert not (tmp_path / "r").exists()
