"""Route matrix: every instantiation of the feature kernels, reached through the call that selects it, against a plain
fp64 evaluation of the same operation.

liblidfe.so compiles fbank_warp_kernel<TIn, kStdMel, kStats>, fbank_kernel<TIn, kMfcc, kStdMel> and
fbank_precise_kernel<TIn, kCenter> for several template arguments.  The input type, the mel bank, the statistics, the
framing, the pad and the alignment choose one of them at run time (route_for in lidfe_abi.cu).  Each row of
ROUTES names a configuration, a call and the exact kernels that call must launch; the GPU test checks that those kernels
ran (torch.profiler) and that what they computed matches the fp64 references of oracle.frontend_oracle:

  * raw features: log-mel rows against the fp32 oracle (metrics (ii)/(iii) of test_gpu_parity.py) and, pooled, no
    worse than it against the fp64 truth (metric (iv)); dB rows 1e-4 of the range from the fp64 truth; MFCC rows 1e-4
    from the oracle and 2e-6 of the range from the device's own log-mels x DCT x lifter in fp64; precise rows the fp64
    truth rounded once;
  * the second stage on the same kernel's raw output: per-utterance CMVN, the top_db clamp (bit exact), global
    accumulate / apply;
  * edges: Kaldi / CENTER lengths at the framing limits, silence, a quiet tail, a DC offset, full-scale int16, an
    eight-row mask table, the padded and the packed layout, and output rows with a leading dimension > n_out.

test_kernel_inventory (CPU) lists the kernels the library holds: a new instantiation without a route fails it."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest
import torch

from oracle import frontend_oracle as O
from test_gpu_parity import _check_fbank, _check_no_worse_than_reference, _cuda_kernels

gpu = pytest.mark.gpu

F32, I16 = "float", "short"
APPLY, DCT, WAVE0 = "cmvn_apply_kernel", "mfcc_dct_mma_kernel", "wave_stages_kernel<0>"
I16_SCALE = 1.0 / 32768.0


def W(t, std_mel, stats):
    return "fbank_warp_kernel<%s, %d, %d>" % (t, std_mel, stats)


def CTA(t, mfcc, std_mel):
    return "fbank_kernel<%s, %s, %d>" % (t, "true" if mfcc else "false", std_mel)


def PR(t, center):
    return "fbank_precise_kernel<%s, %s>" % (t, "true" if center else "false")


def _route(rid, kw, mode, kernels, env=None, raw=False, abi_ceps=0, shift=0):
    """kw: FrontEnd kwargs.  mode: none / utt / accum / apply / topdb (the C ABI's cmvn modes; every call goes through
    lidfe_featurize, so the melspec rows may use the modes FrontEnd.featurize_packed refuses).  env: LIDFE_WARP_KERNEL at
    creation.  raw: lidfe_featurize_raw (normalize_wav fused into the load).  abi_ceps: a melspec handle re-created with
    that many cepstra, which FrontEnd(kind="melspec_db") never builds.  shift: every utterance starts that many samples
    past a 16-byte boundary of the packed buffer."""
    return dict(id=rid, kw=kw, mode=mode, kernels=frozenset(kernels), env=env, raw=raw, abi_ceps=abi_ceps, shift=shift)


_I16 = dict(in_dtype=torch.int16, in_scale=I16_SCALE)
_MEL = dict(kind="melspec_db")
ROUTES = [
    # ---- Kaldi framing, warp-autonomous kernel: <TIn, 1 = Kaldi-80 call, 0 = generic bank, kStats>
    _route("k80", {}, "none", [W(F32, 1, 0)]),
    _route("k80_utt", {}, "utt", [W(F32, 1, 1), APPLY]),
    _route("k80_accum", {}, "accum", [W(F32, 1, 1)]),
    _route("k80_apply", {}, "apply", [W(F32, 1, 0)]),
    _route("k80_i16", _I16, "none", [W(I16, 1, 0)]),
    _route("k80_i16_utt", _I16, "utt", [W(I16, 1, 1), APPLY]),
    _route("k80_i16_scale3000", dict(in_dtype=torch.int16, in_scale=1.0 / 3000.0), "none", [W(I16, 1, 0)]),
    _route("k40", dict(n_mels=40), "none", [W(F32, 0, 0)]),
    _route("k40_utt", dict(n_mels=40), "utt", [W(F32, 0, 1), APPLY]),
    _route("k40_i16", dict(n_mels=40, **_I16), "none", [W(I16, 0, 0)]),
    _route("k40_i16_utt", dict(n_mels=40, **_I16), "utt", [W(I16, 0, 1), APPLY]),
    _route("k40_i16_accum", dict(n_mels=40, **_I16), "accum", [W(I16, 0, 1)]),
    _route("k80_hamming_nodc", dict(window="hamming", remove_dc=False, preemph=0.97), "none", [W(F32, 0, 0)]),
    # ---- Kaldi framing, fbank_kernel: the LIDFE_WARP_KERNEL=0 selector, the fused normalize_wav load, MFCC epilogue
    _route("k80_cta", {}, "none", [CTA(F32, False, 1)], env="0"),
    _route("k80_cta_utt", {}, "utt", [CTA(F32, False, 1), APPLY], env="0"),
    _route("k80_raw", {}, "none", [WAVE0, CTA(F32, False, 1)], raw=True),
    _route("k80_unaligned", {}, "none", [CTA(F32, False, 1)], shift=1),
    _route("k80_dither", dict(dither=0.05, seed=0x1234567811), "none", [CTA(F32, False, 1)]),
    _route("k80_i16_raw", _I16, "none", [WAVE0, CTA(I16, False, 1)], raw=True),
    _route("k40_cta", dict(n_mels=40), "none", [CTA(F32, False, 0)], env="0"),
    _route("k40_i16_cta", dict(n_mels=40, **_I16), "none", [CTA(I16, False, 0)], env="0"),
    _route("mfcc40", dict(n_ceps=40), "none", [W(F32, 1, 0), DCT]),
    _route("mfcc40_i16", dict(n_ceps=40, **_I16), "none", [W(I16, 1, 0), DCT]),
    _route("mfcc40_raw", dict(n_ceps=40), "none", [WAVE0, CTA(F32, False, 1), DCT], raw=True),
    _route("mfcc40_utt", dict(n_ceps=40), "utt", [CTA(F32, True, 1), APPLY]),
    _route("mfcc40_i16_utt", dict(n_ceps=40, **_I16), "utt", [CTA(I16, True, 1), APPLY]),
    _route("mfcc60", dict(n_ceps=60), "none", [CTA(F32, True, 1)]),
    _route("mfcc13_23", dict(n_mels=23, n_ceps=13, preemph=0.97), "none", [CTA(F32, True, 0)]),
    _route("mfcc13_23_i16", dict(n_mels=23, n_ceps=13, preemph=0.97, **_I16), "none", [CTA(I16, True, 0)]),
    # ---- CENTER framing (the reference's default branch): warp kernel <TIn, 2, kStats> when the pad keeps the bulk
    #      copies 16-byte aligned (pad * sizeof(TIn) % 16 == 0), fbank_kernel otherwise and for generic banks
    _route("mel_p0", dict(pad=0, **_MEL), "topdb", [W(F32, 2, 2), APPLY]),
    _route("mel_p16", dict(pad=16, **_MEL), "topdb", [W(F32, 2, 2), APPLY]),
    _route("mel_p300", dict(pad=300, **_MEL), "topdb", [W(F32, 2, 2), APPLY]),
    _route("mel_topdb20", dict(pad=0, top_db=20.0, **_MEL), "topdb", [W(F32, 2, 2), APPLY]),
    _route("mel_p2", dict(pad=2, **_MEL), "topdb", [CTA(F32, False, 2), APPLY]),
    _route("mel_p0_unaligned", dict(pad=0, **_MEL), "topdb", [CTA(F32, False, 2), APPLY], shift=1),
    _route("mel_n64", dict(pad=0, n_mels=64, **_MEL), "topdb", [CTA(F32, False, 0), APPLY]),
    _route("mel_i16_p0", dict(pad=0, **_MEL, **_I16), "topdb", [W(I16, 2, 2), APPLY]),
    _route("mel_i16_p4", dict(pad=4, **_MEL, **_I16), "topdb", [CTA(I16, False, 2), APPLY]),
    _route("mel_i16_p8", dict(pad=8, **_MEL, **_I16), "topdb", [W(I16, 2, 2), APPLY]),
    _route("mel_i16_n64", dict(pad=16, n_mels=64, **_MEL, **_I16), "topdb", [CTA(I16, False, 0), APPLY]),
    _route("mel_abi_none", dict(pad=16, **_MEL), "none", [W(F32, 2, 0)]),
    _route("mel_abi_apply", dict(pad=16, **_MEL), "apply", [W(F32, 2, 0)]),
    _route("mel_abi_utt", dict(pad=0, **_MEL), "utt", [W(F32, 2, 1), APPLY]),
    _route("mel_abi_accum", dict(pad=0, **_MEL), "accum", [W(F32, 2, 1)]),
    _route("mel_abi_i16_none", dict(pad=8, **_MEL, **_I16), "none", [W(I16, 2, 0)]),
    _route("mel_abi_i16_utt", dict(pad=0, **_MEL, **_I16), "utt", [W(I16, 2, 1), APPLY]),
    _route("mel_abi_mfcc60", dict(pad=16, **_MEL), "none", [CTA(F32, True, 2)], abi_ceps=60),
    _route("mel_abi_mfcc40_i16_utt", dict(pad=0, **_MEL, **_I16), "utt", [CTA(I16, True, 2), APPLY], abi_ceps=40),
    # ---- precise mode: the fp64 kernel, both framings
    _route("precise_k80", dict(precise=True), "none", [PR(F32, False)]),
    _route("precise_k80_i16", dict(precise=True, **_I16), "none", [PR(I16, False)]),
    _route("precise_mel", dict(pad=16, precise=True, **_MEL), "topdb", [PR(F32, True), APPLY]),
    _route("precise_mel_i16", dict(pad=4, precise=True, **_MEL, **_I16), "topdb", [PR(I16, True), APPLY]),
]

# every other kernel of the library, with the test that covers it
OTHER_KERNELS = {
    "cmvn_apply_kernel": "tests/test_gpu_dispatch.py (second stage, masks, strided rows)",
    "mfcc_dct_mma_kernel": "tests/test_gpu_dispatch.py, test_gpu_parity.py::test_generic_kernel_variant_configs",
    "resample_kernel": "test_gpu_gemm_routes.py::test_gemm_route",
    "resample_tc_kernel": "test_gpu_gemm_routes.py::test_gemm_route",
    "wave_stages_kernel<0>": "test_gpu_parity.py::test_wave_stages, tests/test_gpu_dispatch.py (raw rows)",
    "wave_stages_kernel<1>": "test_gpu_noise.py (noise bank)",
    "wave_stages_kernel<2>": "test_gpu_noise.py (Gaussian noise)",
    "stft_mel_db_kernel": "test_gpu_gemm_routes.py::test_gemm_route (S3prlFBank rows)",
    "scalar_norm_kernel": "test_gpu_gemm_routes.py::test_gemm_route (S3prlFBank rows)",
    "h2d_gather_kernel": "test_gpu_precise.py::test_h2d_gather_kernel_and_its_fallback",
    "fp32_probe_kernel": "bench roofline probe only",
}


def _canon(name):
    """'void lidfe::fbank_warp_kernel<short, 2, 2>(lidfe::FbankParams)' -> 'fbank_warp_kernel<short,2,2>'"""
    n = name.strip()
    if n.startswith("void "):
        n = n[5:]
    n = re.sub(r"\(.*\)$", "", n).replace("lidfe::", "").replace("(int)", "").replace("(bool)", "")
    return n.replace(" ", "")


def _our_kernels(names):
    names = list(names)
    mangled = [n for n in names if n.startswith("_Z")]
    if mangled and shutil.which("c++filt"):          # a profiler that reports mangled names
        names += subprocess.run(["c++filt"], input="\n".join(mangled), check=True, capture_output=True,
                                text=True).stdout.splitlines()
    return {_canon(n) for n in names if "lidfe::" in n or _canon(n) in OTHER_KERNELS}


def test_kernel_inventory():
    """The library's entry kernels, demangled: the fbank_* ones are exactly the routes' expected kernels, every other one
    is named in OTHER_KERNELS."""
    import speech_lid_b200._lib as L
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("liblidfe.so is not built")
    cands = [os.path.join(d, "bin", "cuobjdump") for d in (os.environ.get("CUDA_HOME"), "/usr/local/cuda") if d]
    cuobjdump = next((c for c in cands if os.path.exists(c)), None) or shutil.which("cuobjdump")
    cxxfilt = shutil.which("c++filt")
    if not cuobjdump or not cxxfilt:
        pytest.skip("cuobjdump or c++filt not found")
    listing = subprocess.run([cuobjdump, "--list-text", L.LIB_PATH], check=True, capture_output=True, text=True).stdout
    mangled = re.findall(r"-(\w+)\.sm_\w+\.elf\.bin", listing)
    demangled = subprocess.run([cxxfilt], input="\n".join(mangled), check=True, capture_output=True, text=True).stdout
    kernels = {_canon(n) for n in demangled.splitlines() if n.strip()}
    print("%d kernels in %s" % (len(kernels), L.LIB_PATH))
    assert len(kernels) == len(mangled)
    routed = set().union(*[{_canon(k) for k in r["kernels"]} for r in ROUTES])
    fbank = {k for k in kernels if k.startswith("fbank_")}
    assert fbank == {k for k in routed if k.startswith("fbank_")}, (
        "instantiations without a route: %s; routes to missing kernels: %s" % (sorted(fbank - routed), sorted(routed - kernels)))
    assert kernels - fbank == set(OTHER_KERNELS), (sorted(kernels - fbank - set(OTHER_KERNELS)),
                                                   sorted(set(OTHER_KERNELS) - kernels))
    assert routed <= kernels


# ------------------------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------------------------
KALDI_BATCH = [(400, "noise"), (401, "speech"), (559, "dc"), (560, "noise"), (561, "speech"), (12347, "full"),
               (16000, "zeros"), (48000, "tail"), (320000, "noise")]          # 12347 = 3 mod 8; 320000 = 20 s


def _center_batch(pad):
    return [(max(1, 257 - 2 * pad), "noise"), (300, "speech"), (2560, "zeros"), (12345, "dc"), (128000, "tail"),
            (16000, "full")]


def _content(kind, n, seed, int16):
    """(1, n) float32 samples, or int16 PCM.  tail: the last quarter 100 dB down.  full: int16 at full scale, the
    extremes +-32767 / -32768 included (clipped noise for float input)."""
    if kind == "zeros":
        return torch.zeros(1, n, dtype=torch.int16 if int16 else torch.float32)
    if n < 64:
        x = torch.randn(1, n, generator=torch.Generator().manual_seed(seed))
    elif kind == "speech":
        x = O.synth_speechlike(n, seed)
    else:
        x = O.synth_noise(n, seed)
    if kind == "dc":
        x = x + 0.5
    if kind == "full":
        x = (x * 0.7).clamp(-1.0, 1.0)
    if kind == "tail":
        x = x.clone()
        x[:, 3 * n // 4:] *= 1e-5
    if not int16:
        return x
    scale = {"full": 32768.0, "tail": 8000.0}.get(kind, 3000.0)
    q = (x.double() * scale).round().clamp(-32768, 32767)
    if kind == "full":
        q[0, 0:n:97] = 32767
        q[0, 1:n:97] = -32768
        q[0, 2:n:97] = -32767
    return q.to(torch.int16)


def _inputs(route, fe):
    int16 = fe.in_dtype == torch.int16
    center = route["kw"].get("kind") == "melspec_db"
    batch = _center_batch(int(route["kw"].get("pad", 0))) if center else KALDI_BATCH
    return [_content(k, n, 4000 + i, int16) for i, (n, k) in enumerate(batch)], [k for _, k in batch]


# ------------------------------------------------------------------------------------------------------------------
# front-ends and calls
# ------------------------------------------------------------------------------------------------------------------
_FE_CACHE = {}


def _frontend(lid, route, **over):
    kw = dict(route["kw"], **over)
    key = (repr(sorted(kw.items(), key=lambda kv: kv[0])), route["env"], route["abi_ceps"])
    if key in _FE_CACHE:
        return _FE_CACHE[key]
    old = os.environ.get("LIDFE_WARP_KERNEL")
    if route["env"] is not None:
        os.environ["LIDFE_WARP_KERNEL"] = route["env"]
    try:
        fe = lid.FrontEnd(**kw)
        if route["abi_ceps"]:
            _add_cepstra(lid, fe, route["abi_ceps"])
    finally:
        if old is None:
            os.environ.pop("LIDFE_WARP_KERNEL", None)
        else:
            os.environ["LIDFE_WARP_KERNEL"] = old
    _FE_CACHE[key] = fe
    return fe


def _add_cepstra(lid, fe, n_ceps):
    """Replace fe's handle by one of the same configuration with n_ceps cepstra (DCT + lifter epilogue)."""
    from speech_lid_b200 import _lib, tables
    cfg = _lib.LidfeConfig.from_buffer_copy(fe.cfg)
    cfg.n_ceps = n_ceps
    window, banks = fe._tables[:2]
    dct = tables.dct_matrix(n_ceps, fe.n_mels).contiguous()
    lift = tables.lifter(n_ceps, 22.0).contiguous()
    h = C.c_void_p()
    _lib.check(fe.lib.lidfe_create(C.byref(h), C.byref(cfg), window.data_ptr(), banks.data_ptr(), dct.data_ptr(),
                                   lift.data_ptr()))
    fe.lib.lidfe_destroy(fe.handle)
    fe.handle, fe.cfg, fe._tables = h.value, cfg, (window, banks, dct, lift)
    fe.n_ceps = fe.n_out = n_ceps
    if fe.precise:
        _lib.check(fe.lib.lidfe_set_precision(fe.handle, 1))


def _modes():
    from speech_lid_b200 import _lib
    return {"none": _lib.CMVN_NONE, "utt": _lib.CMVN_PER_UTT, "apply": _lib.CMVN_APPLY_GLOBAL,
            "accum": _lib.CMVN_ACCUM_GLOBAL, "topdb": _lib.POST_TOPDB}


def _plan(fe, route, lens, padded):
    """fe.make_plan; a route with a shift starts every utterance that many samples past its 16-byte boundary."""
    if not route["shift"]:
        return fe.make_plan(lens, padded=padded)
    offsets, pos = [], 0
    for n in lens:
        offsets.append(pos + route["shift"])
        pos += (route["shift"] + n + fe.align - 1) // fe.align * fe.align
    return fe.make_plan(lens, padded=padded, offsets=offsets)


def _call(fe, route, plan, packed, mode, ld=None, out=None, masks=None, stats_in=None, stats_out=None):
    """One lidfe_featurize(_raw) call; returns the (rows, ld) output."""
    from speech_lid_b200 import _lib
    ld = ld or fe.n_out
    if out is None:
        out = torch.empty(plan.rows * ld, dtype=torch.float32, device=fe.device)
    if mode == "accum" and stats_out is None:
        stats_out = torch.zeros(2 * fe.n_out + 1, dtype=torch.float64, device=fe.device)
    fn = fe.lib.lidfe_featurize_raw if route["raw"] else fe.lib.lidfe_featurize
    ptr = lambda t: None if t is None else t.data_ptr()        # noqa: E731
    _lib.check(fn(fe.handle, plan.handle, packed.data_ptr(), out.data_ptr(), ld, ptr(masks),
                  0 if masks is None else masks.shape[1], _modes()[mode], ptr(stats_in), ptr(stats_out),
                  torch.cuda.current_stream(fe.device).cuda_stream))
    return out.view(plan.rows, ld)


def _rows(out, plan, i):
    return out[plan.out_rows[i]:plan.out_rows[i] + plan.frames[i]]


# ------------------------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------------------------
def _scaled(x, fe):
    """The samples the kernel frames, fp32 (int16 PCM times the configuration's fp32 in_scale)."""
    return x.float() * fe.cfg.in_scale if x.dtype == torch.int16 else x


def _normalize64(x):
    x = x.double()
    std, mean = torch.std_mean(x, dim=-1)
    return (x - mean) / (std + 1e-6)


def _references(route, fe, x):
    """(oracle32, truth64) of the raw features (no second stage) of x under this route's configuration."""
    kw = route["kw"]
    n_mels = fe.n_mels
    w32 = _scaled(x, fe)
    if kw.get("kind") == "melspec_db":
        pad = int(kw.get("pad", 0))
        ref = O.melspec_db(w32, pad=pad, top_db=None, n_mels=n_mels)[0].T
        tru = O.truth64_melspec_db(w32.double(), pad=pad, top_db=None, n_mels=n_mels)
    else:
        args = dict(n_mels=n_mels, preemph=float(kw.get("preemph", 1.0)), window_type=kw.get("window", "povey"),
                    remove_dc=bool(kw.get("remove_dc", True)))
        if route["raw"]:
            ref = O.kaldi_fbank(O.normalize_wav(w32), **args)
            tru = O.truth64_fbank(_normalize64(w32.double() if x.dtype != torch.int16 else x.double() * fe.cfg.in_scale),
                                  **args)
        else:
            ref = O.kaldi_fbank(w32, **args)
            tru = O.truth64_fbank(x, in_scale=fe.cfg.in_scale if x.dtype == torch.int16 else 1.0, **args)
    if fe.n_ceps:
        dct, lift = O.kaldi_dct_matrix(fe.n_ceps, n_mels), O.kaldi_lifter(fe.n_ceps, 22.0)
        ref = ref.matmul(dct) * lift.unsqueeze(0).to(torch.float32)
        tru = (tru @ dct.double()) * lift.double()
    return ref, tru


def _norm_rel(got, want):
    return float((got.double() - want.double()).abs().max() / want.double().abs().max())


def _check_raw(lid, route, fe, wavs, kinds, plan, packed, raw):
    """raw: (rows, n_out) raw features of the route's kernel on the padded plan."""
    kw = route["kw"]
    melspec = kw.get("kind") == "melspec_db"
    triples = []
    lin = None
    if fe.n_ceps and not kw.get("precise"):
        # the device's own log-mels (same configuration without cepstra) x DCT x lifter in fp64
        fb_route = dict(route, abi_ceps=0, kw={k: v for k, v in kw.items() if k != "n_ceps"})
        fb = _frontend(lid, fb_route)
        plan_f = _plan(fb, fb_route, plan.lengths, True)
        logmel = _call(fb, fb_route, plan_f, packed, "none").double()
        from speech_lid_b200 import tables
        lin = (logmel @ tables.dct_matrix(fe.n_ceps, fe.n_mels).to(fe.device).double()) * \
            tables.lifter(fe.n_ceps, 22.0).to(fe.device).double()
        lin = lin.cpu()
    if kw.get("dither"):
        # in-kernel dither: the references see wav + dither * U, U the device's own draw (as in test_gpu_round2.py)
        u = fe.wave_stages(torch.zeros(plan.total_samples, device=fe.device), plan, dither=1.0).cpu()
        amp = torch.tensor(kw["dither"], dtype=torch.float32)
        wavs = [x + amp * u[o:o + x.shape[-1]] for x, o in zip(wavs, plan.offsets)]
    for i, (x, kind) in enumerate(zip(wavs, kinds)):
        got = _rows(raw, plan, i).cpu()
        what = "%s utt %d (%s, %d samples)" % (route["id"], i, kind, x.shape[-1])
        assert torch.isfinite(got).all(), what
        ref, tru = _references(route, fe, x)
        assert got.shape == ref.shape == tru.shape, (what, got.shape, ref.shape)
        if kind == "zeros" and not fe.n_ceps and not kw.get("dither"):
            floor = -100.0 if melspec else float(torch.tensor(O.EPS32).log())
            assert torch.all(got == floor), "%s: silence is not exactly %r" % (what, floor)
            assert torch.equal(got, ref), what
        if kw.get("precise"):
            bound = 4e-6 if fe.n_ceps else (1e-5 if melspec else 1e-6)
            assert float((got.double() - tru).abs().max()) <= bound, (what, float((got.double() - tru).abs().max()))
        elif fe.n_ceps:
            assert _norm_rel(got, ref) <= 1e-4, (what, _norm_rel(got, ref))
            rel = float((got.double() - _rows(lin, plan, i)).abs().max() / _rows(lin, plan, i).abs().max())
            assert rel <= 2e-6, (what, rel)
        elif melspec:
            assert _norm_rel(got, tru) <= 1e-4, (what, _norm_rel(got, tru))
            assert _norm_rel(got, ref) <= 1e-4, (what, _norm_rel(got, ref))
        else:
            if kind == "tail":      # the quiet quarter is judged against its own bin medians (see _deep_nulls)
                q = max(0, (3 * x.shape[-1] // 4 - 400) // 160 + 1)
                _check_fbank(got[:q], ref[:q], what + " loud part")
                _check_fbank(got[q:], ref[q:], what + " quiet tail")
            else:
                _check_fbank(got, ref, what, all_bins=(kind == "speech"))
            triples.append((got, ref, tru))
    if triples:
        _check_no_worse_than_reference(triples, route["id"])


def _assert_close_or_equal(a, b, tol, what):
    """Bit-equal (NaNs in the same places) when tol == 0, else |a - b| <= tol."""
    a, b = a.cpu(), b.cpu()
    assert torch.equal(torch.isnan(a), torch.isnan(b)), what
    a, b = torch.nan_to_num(a, nan=0.0), torch.nan_to_num(b, nan=0.0)
    if tol == 0:
        assert torch.equal(a, b), (what, float((a - b).abs().max()))
    else:
        assert float((a - b).abs().max()) <= tol, (what, float((a - b).abs().max()))


def _edge_masks(frames, n_out, full_utt):
    """Eight rows per utterance (more than cmvn_apply_kernel's four register masks), every bound in [0,T] x [0,n_out]:
    the first cell, the last cell, empty time / frequency ranges, and one utterance masked entirely."""
    rows = []
    for i, T in enumerate(frames):
        r = [(0, 1, 0, 1), (T - 1, T, n_out - 1, n_out), (T // 2, T // 2, 2, 5), (min(1, T), min(3, T), 7, 7),
             (0, 0, 0, 0), (T // 3, T // 3 + 1, n_out // 2, n_out // 2 + 1), (T, T, n_out, n_out),
             (0, T, 0, n_out) if i == full_utt else (T // 4, T // 4, 0, 0)]
        rows.append(r)
    return torch.tensor(rows, dtype=torch.int32)


SENTINEL = 0x7FC0DEAD           # a quiet-NaN payload no kernel writes


@pytest.fixture(scope="module")
def lid():
    import speech_lid_b200 as m
    return m


@gpu
@pytest.mark.parametrize("route", ROUTES, ids=[r["id"] for r in ROUTES])
def test_route(lid, route):
    fe = _frontend(lid, route)
    wavs, kinds = _inputs(route, fe)
    lens = [int(w.shape[-1]) for w in wavs]
    mode = route["mode"]
    stat_mode = mode in ("utt", "accum")          # fp64 atomics: the sums' order varies between launches
    tol = 2e-6 if stat_mode else 0.0
    plan = _plan(fe, route, lens, True)
    plan_p = _plan(fe, route, lens, False)
    assert plan.frames == [fe.num_frames(n) for n in lens]
    packed = fe.pack(wavs, plan)
    packed_p = fe.pack(wavs, plan_p)

    # ---- raw features of the route's own kernel, and the statistics / clamp inputs of its second stage
    stats_in = None
    if mode in ("none", "accum"):
        raw = None
    elif mode == "utt":
        raw = _call(fe, route, plan, packed, "accum")
    elif mode == "topdb":
        fe_inf = _frontend(lid, route, top_db=float("inf"))      # same kernel; the clamp never bites
        raw = _call(fe_inf, route, _plan(fe_inf, route, lens, True), packed, "topdb")
    else:       # apply
        raw = _call(fe, route, plan, packed, "none")
        stats_in = O.cmvn_stats([_rows(raw, plan, i).cpu() for i in range(len(lens))]).to(fe.device)

    # ---- dispatch, padded and packed layouts
    expected = {_canon(k) for k in route["kernels"]}
    outs = {}
    for layout, pl, pk in (("padded", plan, packed), ("packed", plan_p, packed_p)):
        so = torch.zeros(2 * fe.n_out + 1, dtype=torch.float64, device=fe.device) if mode == "accum" else None
        out, names = _cuda_kernels(lambda: _call(fe, route, pl, pk, mode, stats_in=stats_in, stats_out=so))
        ran = _our_kernels(names)
        if ran != expected:
            print("%s (%s) launched: %s" % (route["id"], layout, sorted(names)))
        assert ran == expected, (route["id"], layout, sorted(ran), sorted(expected))
        outs[layout] = (out, so)
    out, stats = outs["padded"]
    for i in range(len(lens)):
        _assert_close_or_equal(_rows(outs["packed"][0], plan_p, i), _rows(out, plan, i), tol,
                               "%s: packed vs padded, utt %d" % (route["id"], i))
        assert torch.all(out[plan.out_rows[i] + plan.frames[i]:plan.out_rows[i] + plan.t_max] == 0)
    if raw is None:
        raw = out

    # ---- raw features against the fp32 oracle and the fp64 truth
    _check_raw(lid, route, fe, wavs, kinds, plan, packed, raw)

    # ---- second stage against fp64 on the kernel's own raw output
    raw_c, out_c = raw.cpu(), out.cpu()
    if mode == "utt":
        for i, kind in enumerate(kinds):
            want = O.cmvn_per_utt(_rows(raw_c, plan, i))
            got = _rows(out_c, plan, i)
            assert torch.allclose(got, want, rtol=1e-5, atol=2e-6, equal_nan=True), (route["id"], i, kind)
            if kind == "zeros" and plan.frames[i] > 1:
                assert torch.all(got == 0), "%s: CMVN of silence must be exactly 0" % route["id"]
    elif mode == "topdb":
        top_db = torch.tensor(float(route["kw"].get("top_db", 80.0)), dtype=torch.float32)
        for i, kind in enumerate(kinds):
            r = _rows(raw_c, plan, i)
            assert torch.equal(_rows(out_c, plan, i), torch.maximum(r, r.max() - top_db)), (route["id"], i)
            if kind == "zeros":
                assert torch.all(_rows(out_c, plan, i) == -100.0)
        t = kinds.index("tail")      # the clamp bites in the quiet tail
        assert float(_rows(out_c, plan, t).min()) == float(_rows(raw_c, plan, t).max() - top_db)
    elif mode == "accum":
        rows = [_rows(raw_c, plan, i) for i in range(len(lens))]
        assert float(stats[-1]) == sum(plan.frames)
        assert torch.allclose(stats.cpu(), O.cmvn_stats(rows), rtol=1e-6, atol=1e-4)
        assert torch.allclose(outs["packed"][1].cpu(), O.cmvn_stats(rows), rtol=1e-6, atol=1e-4)
    elif mode == "apply":
        mean, std = O.cmvn_finalize(stats_in.cpu())
        for i in range(len(lens)):
            want = O.cmvn_apply(_rows(raw_c, plan, i), mean, std)
            assert torch.allclose(_rows(out_c, plan, i), want, rtol=1e-5, atol=2e-6), (route["id"], i)

    # ---- masks at the edges (the accumulate mode takes none)
    if mode != "accum":
        masks = _edge_masks(plan.frames, fe.n_out, full_utt=kinds.index("noise")).to(fe.device)
        masked = _call(fe, route, plan, packed, mode, masks=masks, stats_in=stats_in).cpu()
        for i in range(len(lens)):
            b = [tuple(int(v) for v in masks[i, q]) for q in range(masks.shape[1])]
            want = O.apply_mask_bounds(_rows(out_c, plan, i).T.unsqueeze(0), b)[0].T
            got = _rows(masked, plan, i)
            hole = O.apply_mask_bounds(torch.ones_like(want).T.unsqueeze(0), b)[0].T == 0
            assert torch.all(got[hole] == 0), (route["id"], i)
            _assert_close_or_equal(got, want, tol, "%s: masked call, utt %d" % (route["id"], i))
        assert torch.all(_rows(masked, plan, kinds.index("noise")) == 0)

    # ---- output rows with a leading dimension > n_out: the columns past n_out keep the sentinel
    n = fe.n_out
    for ld in (n + 1, n + 4):
        buf = torch.full((plan.rows * ld,), SENTINEL, dtype=torch.int32, device=fe.device)
        so = torch.zeros(2 * n + 1, dtype=torch.float64, device=fe.device) if mode == "accum" else None
        got = _call(fe, route, plan, packed, mode, ld=ld, out=buf.view(torch.float32), stats_in=stats_in, stats_out=so)
        gi = got.view(torch.int32).cpu()
        assert torch.all(gi[:, n:] == SENTINEL), (route["id"], ld)
        if tol == 0:
            assert torch.equal(gi[:, :n], out.view(torch.int32).cpu()), (route["id"], ld)
        else:
            _assert_close_or_equal(got[:, :n], out, tol, "%s: ld %d" % (route["id"], ld))
