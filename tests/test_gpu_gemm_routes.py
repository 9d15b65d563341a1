"""Route matrix of the windowed-GEMM family: the polyphase resampler (`Resampler`) and the wav2vec-exp FBank variant
(`S3prlFBank`), at every tiling their kernels run, against plain fp64 evaluations of the same operations.

lidfe_resample runs one of two kernels.  resample_tc_kernel (tcgen05, accumulators in TMEM, an mbarrier pipeline) takes
every bank whose row count nw is a multiple of 16; resample_kernel (FP32) takes the others and every bank created under
LIDFE_RESAMPLE_TC=0.  create_bank (lidfe_abi.cu) fixes the tensor-core tiling: N phases per tile, nw / N phase tiles, KB
32-tap blocks, a pipeline of `stages` blocks.  The kernel is persistent -- grid = min(linear tiles, SMs), a CTA walks tiles
L, L + grid, ... -- and only from a CTA's second live tile on do the two TMEM accumulator buffers alternate, the MMA warp
wait on acc_empty (third tile) and the builder warps carry pipeline items across tile boundaries.  Each row of ROWS
names a constructor, the kernels its calls must launch and the tiling tc_tiling() derives from create_bank's rule; each
row runs an edge batch (framing limits, silence, DC, full scale, a quiet tail, odd input offsets) and a walk batch sized
from the device's SM count so that some CTA takes at least three live tiles (tile_live() restates the kernel's
linearisation).

Checks: every output sample of the GEMM within GEMM_C U sum_k |w_k x_k| + 2 U sum |running sum| of the fp64 sum (see
GEMM_C); the S3prl chain stage by stage (GEMM rows, power -> mel -> dB on the device's own GEMM output, the scalar
normalisation on the device's own dB rows) and end to end against oracle.frontend_oracle.truth64_s3prl_fbank, no worse
than a model of the kernel's arithmetic (gemm_terms, model_chain); the tensor-core kernel against the FP32 one; writes
that stay inside out_off / out_len.  The CPU tests pin the tiling rule, the matrix's coverage, and that the bounds reject
emulated kernel mistakes.  The GPU part of this file takes about 18 s on a B200."""
import math
import os

import pytest
import torch

from oracle import frontend_oracle as O
from test_gpu_dispatch import SENTINEL, _content, _our_kernels
from test_gpu_parity import _cuda_kernels

gpu = pytest.mark.gpu

U = 2.0 ** -24
# |y - sum_k w_k x_k| <= GEMM_C U sum_k |w_k x_k| + 2 U acc per output sample (gemm_ratio, gemm_terms).
#  * products: resample_tc_kernel splits both operands into hi = tf32(v) (round to nearest) and lo = v - hi, which the
#    tensor core reads truncated to tf32, and drops lo * lo: each product loses at most (2^-21 + 2^-21 + 2^-22) |w x|
#    = 20 U |w x|.  GEMM_C = 32 covers that worst case with room for the rounding inside an instruction's sum.
#  * accumulation: per 8 taps the kernel issues three MMAs into the fp32 accumulator in TMEM, and the tensor core rounds
#    each update toward zero, so it loses up to one ulp (2 U) of the running sum, always toward zero; acc sums the
#    |running sum| over those updates.  On input whose partial sums share a sign (a periodic frame, a DFT bin near DC)
#    the losses add up (K / 8 ulps at most) instead of cancelling; where they do not, acc stays small and so does the
#    bound.  resample_kernel's chain of fmaf (round to nearest) stays far inside it.
# The modelled kernel uses 0.4 of the bound; one TF32 pass or a dropped correction term exceeds it 15 to 130 times, a
# wrong tap block or phase by orders of magnitude (test_bounds_reject_emulated_kernel_mistakes).
GEMM_C = 32.0
DB_PER_REL = 10.0 / math.log(10.0)         # d(10 log10 p) / (dp / p)

TC, FP32, MELDB, NORM = "resample_tc_kernel", "resample_kernel", "stft_mel_db_kernel", "scalar_norm_kernel"
TC_M, TC_KB, TC_ABYTES = 128, 32, 128 * 32 * 4     # lidfe_resample_tc.cuh: kTcM, kTcKB, kTcABytes


def tc_tiling(nw, taps):
    """create_bank's rule (lidfe_abi.cu) restated: (N, phase tiles, KB, stages) of resample_tc_kernel, or None when the
    bank goes to resample_kernel.  N is the largest multiple of 32 <= 256 that divides nw, else the largest such
    multiple of 16; KB = max(2, ceil(taps / 32)); as many stages of 2 (A + B) images as fit 220 KB, at most 4 and KB."""
    N = next((c for c in range(256, 31, -32) if nw % c == 0), 0) or next((c for c in range(240, 15, -16) if nw % c == 0), 0)
    if N == 0:
        return None
    KB = max(2, -(-taps // TC_KB))
    stage = 2 * TC_ABYTES + 2 * N * 128
    return N, nw // N, KB, min(4, (220 * 1024) // stage, KB)


def tile_live(out_len, nw, n_tiles, max_out_len):
    """resample_tc_kernel's linearisation (tile_live in lidfe_resample_tc.cuh): linear tile L is (phase tile
    L / (gx B), utterance (L / gx) % B, frame tile L % gx), live when its first frame lies inside the utterance's output.
    Returns the live flag of every linear tile."""
    frames = -(-max_out_len // nw)
    gx = -(-frames // TC_M)
    B = len(out_len)
    L = torch.arange(gx * B * n_tiles)
    bb = (L // gx) % B
    f0 = (L % gx) * TC_M
    return f0 * nw < torch.tensor(out_len, dtype=torch.long)[bb]


def tiles_per_cta(live, sms):
    """Live tiles each persistent CTA walks (grid = min(linear tiles, SMs), CTA c takes c, c + grid, ...)."""
    grid = min(live.numel(), sms)
    per = torch.zeros(grid, dtype=torch.long).index_add_(0, torch.arange(live.numel()) % grid, live.long())
    return per


# ------------------------------------------------------------------------------------------------------------------
# the matrix
# ------------------------------------------------------------------------------------------------------------------
def _rs(orig, new, kernel, tiling=None, nw=None, env=None):
    rid = "rs_%d_%d%s" % (orig, new, "_fp32sel" if env else "")
    return dict(id=rid, kind="rs", orig=orig, new=new, env=env, kernels=frozenset(kernel), tiling=tiling, nw=nw)


def _s3(fbank_size, n_fft, tiling):
    return dict(id="s3_%d_%d" % (fbank_size, n_fft), kind="s3", fbank_size=fbank_size, n_fft=n_fft, env=None,
                kernels=frozenset([TC, MELDB, NORM]), tiling=tiling, nw=None)


_TC_RATES = [(44100, 16000, (160, 1, 15, 3)), (22050, 16000, (160, 2, 15, 3)), (11025, 16000, (160, 4, 15, 3)),
             (25000, 16000, (16, 1, 2, 2)), (15000, 16000, (16, 1, 2, 2)), (88200, 16000, (80, 1, 16, 4)),
             (44100, 48000, (160, 1, 6, 3))]
ROWS = (
    # ---- Resampler, tcgen05: (N, phase tiles, KB, stages)
    [_rs(o, n, [TC], tiling=t) for o, n, t in _TC_RATES] +
    # ---- Resampler, FP32: the same rates under the selector, then every rate whose reduced new rate is no multiple of 16
    [_rs(o, n, [FP32], nw=t[0] * t[1], env="0") for o, n, t in _TC_RATES] +
    [_rs(o, n, [FP32], nw=nw) for o, n, nw in [(48000, 16000, 1), (32000, 16000, 1), (24000, 16000, 2),
                                                (96000, 16000, 1), (8000, 16000, 2), (16000, 44100, 441),
                                                (16000, 48000, 3)]] +
    # ---- S3prlFBank: windowed-DFT GEMM on the tensor cores, then stft_mel_db_kernel and scalar_norm_kernel
    [_s3(80, n, t) for n, t in [(4, (32, 1, 2, 2)), (16, (32, 1, 2, 2)), (64, (96, 1, 2, 2)), (320, (192, 2, 10, 2)),
                                (400, (224, 2, 13, 2)), (480, (256, 2, 15, 2)), (500, (256, 2, 16, 2)),
                                (512, (192, 3, 16, 2)), (640, (224, 3, 20, 2)), (1024, (224, 5, 32, 2)),
                                (2048, (160, 13, 64, 3))]] +
    [_s3(f, 640, (224, 3, 20, 2)) for f in (1, 40, 128)]
)


def _geometry(row):
    """(bank fp32 (nw, taps), hop, left pad) of the row's GEMM, built by the package's own table code."""
    from speech_lid_b200 import tables
    if row["kind"] == "rs":
        kernel, width = tables.sinc_resample_kernel(row["orig"], row["new"])
        g = math.gcd(row["orig"], row["new"])
        return kernel, row["orig"] // g, width
    bank, _ = tables.windowed_dft_bank(row["n_fft"])
    return bank, row["n_fft"] // 2, 0


def test_tiling_rule_gives_each_rows_tiling():
    """Each row's stated tiling is what create_bank's rule gives its bank; a row without one goes to resample_kernel."""
    for row in ROWS:
        bank, hop, left = _geometry(row)
        nw, taps = bank.shape
        got = tc_tiling(nw, taps)
        if row["env"] == "0" or FP32 in row["kernels"]:
            assert row["tiling"] is None and row["nw"] == nw, row["id"]
            if row["env"] is None:
                assert got is None, row["id"]            # no multiple of 16: the FP32 kernel is the only path
            else:
                assert got is not None, row["id"]        # the selector is what keeps the tensor cores out
        else:
            assert got == row["tiling"], (row["id"], got, row["tiling"])
    # the issue's table of shapes, and the layout constants tc_tiling leans on
    assert tc_tiling(2080, 2048) == (160, 13, 64, 3) and tc_tiling(80, 509) == (80, 1, 16, 4)
    assert tc_tiling(16, 29) == (16, 1, 2, 2) and tc_tiling(441, 174) is None


def test_matrix_coverage():
    """N, phase tiles, KB and stages that the tensor-core kernel can take all appear, and the FP32 kernel runs one phase,
    a few, and more phases than its 160 threads (441 = 160 + 160 + 121, a partial last pass)."""
    tilings = [r["tiling"] for r in ROWS if r["tiling"] is not None]
    assert {t[0] for t in tilings} == {16, 32, 80, 96, 160, 192, 224, 256}
    tiles = {t[1] for t in tilings}
    assert min(tiles) == 1 and max(tiles) == 13 and {1, 2, 3, 4, 5, 13} <= tiles
    assert 2 in {t[2] for t in tilings} and any(t[2] % 2 for t in tilings)
    assert {t[3] for t in tilings} == {2, 3, 4}
    assert {r["nw"] for r in ROWS if FP32 in r["kernels"]} >= {1, 2, 3, 441}
    s3 = {(r["fbank_size"], r["n_fft"]) for r in ROWS if r["kind"] == "s3"}
    assert {n for _, n in s3} >= {4, 16, 64, 320, 400, 500, 512, 640, 1024, 2048}
    assert {f for f, n in s3 if n == 640} == {1, 40, 80, 128}
    # the rows the walk batch must drive through both accumulator buffers: odd KB at N = 160, and N = 224
    assert any(r["tiling"] == (160, 1, 15, 3) and r["kind"] == "rs" for r in ROWS)
    assert any(r["tiling"][0] == 224 and r["kind"] == "s3" and r["n_fft"] == 640 for r in ROWS if r["tiling"])


# ------------------------------------------------------------------------------------------------------------------
# batches
# ------------------------------------------------------------------------------------------------------------------
def _edge_batch(row, hop):
    """(length, content) pairs: the framing limits of the row's kernel and every special content."""
    if row["kind"] == "rs":
        lens = [1, 37 * hop + 5, TC_M * hop - 1, TC_M * hop, TC_M * hop + 1, (3 * TC_M + 50) * hop + 7, 2, hop]
    else:
        n = row["n_fft"]
        frames = lambda f: n + (f - 1) * hop          # noqa: E731
        lens = [n, n + 1, frames(37) + 7, frames(TC_M) - 1, frames(TC_M), frames(TC_M) + 1, frames(3 * TC_M + 50) + 3,
                frames(2)]
    kinds = ["speech", "dc", "full", "zeros", "tail", "noise", "zeros", "speech"]
    return list(zip(lens, kinds))


def _walk_lengths(row, hop, n_tiles, sms):
    """Six ragged utterances with about 3.5 live tiles per SM in all: some CTA walks at least three."""
    per = max(1, -(-(7 * sms // 2) // (6 * n_tiles)))            # frame tiles per utterance
    lens = []
    for i in range(6):
        frames = max(1, per + i % 3 - 1) * TC_M - (37 * i) % 100
        lens.append(frames * hop if row["kind"] == "rs" else row["n_fft"] + (frames - 1) * hop + i % hop)
    return lens


def _pack(wavs, dev):
    """Odd input offsets, with 1e6 in the gaps: a read outside an utterance shows as a gross error."""
    offs, pos = [], 1
    for w in wavs:
        offs.append(pos)
        pos += w.numel() + (2 if (pos + w.numel()) % 2 else 3)
    buf = torch.full((pos + 1,), 1e6, dtype=torch.float32, device=dev)
    for o, w in zip(offs, wavs):
        buf[o:o + w.numel()] = w.to(dev)
    return buf, offs


# ------------------------------------------------------------------------------------------------------------------
# references and bounds (also run on emulated kernels by the CPU tests)
# ------------------------------------------------------------------------------------------------------------------
def _rz(v):
    """float64 -> fp32 rounded toward zero."""
    r = v.float()
    return torch.where(r.double().abs() > v.abs(), torch.nextafter(r, torch.zeros_like(r)), r)


def gemm_terms(x, bank, hop, left, passes=0, chunk=4096):
    """The GEMM of the frames of x (hop apart, `left` zeros in front) with bank, per K = 8 step of taps as the tensor core
    takes it.  Returns (want, mag, acc, model), each (frames, nw):
      want  sum_k w_k x_k in float64,
      mag   sum_k |w_k x_k|,
      acc   the sum of |running sum| over the accumulator updates resample_tc_kernel makes: three per step (lo.hi, hi.lo,
            hi.hi), the first two of which leave it at the previous step's value,
      model (passes > 0) the kernel's arithmetic: hi = tf32_rna(v), lo = v - hi read truncated to tf32; per step
            D += x_lo.w_hi, D += x_hi.w_lo, D += x_hi.w_hi (passes 3; 2 drops x_lo.w_hi, 1 keeps x_hi.w_hi), each
            product sum exact and each update of the fp32 accumulator D rounded toward zero."""
    K, nw = bank.shape[1], bank.shape[0]
    J = -(-K // 8)
    b = torch.nn.functional.pad(bank.to(x.device).float(), (0, 8 * J - K))
    b64 = b.double()
    fr_all = torch.nn.functional.pad(x.float(), (left, left + hop)).unfold(0, K, hop)
    bh = _tf32_rna(b)
    bl = _tf32_trunc(b - bh)
    out = [[], [], [], []]
    for t0 in range(0, fr_all.shape[0], chunk):
        fr = torch.nn.functional.pad(fr_all[t0:t0 + chunk], (0, 8 * J - K))
        f64 = fr.double()
        out[0].append(f64 @ b64.T)
        out[1].append(f64.abs() @ b64.abs().T)
        S = torch.zeros(fr.shape[0], nw, dtype=torch.float64, device=x.device)
        acc = torch.zeros_like(S)
        if passes:
            fh = _tf32_rna(fr)
            fl = _tf32_trunc(fr - fh).double()
            fh = fh.double()
            steps = [(fl, bh.double()), (fh, bl.double()), (fh, bh.double())][3 - passes:]
            D = torch.zeros(fr.shape[0], nw, dtype=torch.float32, device=x.device)
        for j in range(J):
            k = slice(8 * j, 8 * j + 8)
            acc += 2 * S.abs()
            S += f64[:, k] @ b64[:, k].T
            acc += S.abs()
            if passes:
                for a_, b_ in steps:
                    D = _rz(D.double() + a_[:, k] @ b_[:, k].T)
        out[2].append(acc)
        out[3].append(D if passes else None)
    cat = lambda v: torch.cat(v) if v and v[0] is not None else None     # noqa: E731
    return tuple(cat(v) for v in out)


def gemm_ratio(got, want, mag, acc):
    """max of |got - want| / (GEMM_C U mag + 2 U acc); an output whose terms are all zero must be exactly zero (ratio inf
    if not)."""
    err = (got.double() - want).abs()
    lim = GEMM_C * U * mag + 2 * U * acc
    r = torch.where(lim > 0, err / lim.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    return float(r.max()) if r.numel() else 0.0


def mel_db64(g_rows, n_bins, melT):
    """float64 power -> mel -> dB of GEMM rows (re, im interleaved)."""
    z = g_rows.double()[:, :2 * n_bins].reshape(-1, n_bins, 2)
    p = z[..., 0] ** 2 + z[..., 1] ** 2
    return 10.0 * torch.log10((p @ melT.double().T).clamp_min(1e-10))


def model_chain(g_model, n_bins, melT):
    """(dB, normalised) rows of the S3prl chain run on the modelled GEMM rows (gemm_terms(..., passes=3)): power, mel and
    dB in fp32 as stft_mel_db_kernel computes them; scalar_norm_kernel's arithmetic: float64 statistics, then
    ((x - mean32) - (mean - mean32)) * fp32(1 / (std + 1e-9)) with every step in fp32."""
    z = g_model[:, :2 * n_bins].float().reshape(-1, n_bins, 2)
    p = torch.addcmul(z[..., 1] * z[..., 1], z[..., 0], z[..., 0])
    db = 10.0 * torch.log10((p @ melT.float().T).clamp_min(1e-10))
    std, mean = torch.std_mean(db.double())
    mean32 = mean.float()
    lo, inv = (mean - mean32.double()).float(), (1.0 / (std + 1e-9)).float()
    return db, ((db - mean32) - lo) * inv


def mel_db_bound(db64, mel_lo, mel_hi):
    """stft_mel_db_kernel in fp32: the power (one fmaf) and each term of the mel sum (a chain of fmaf over the filter's
    n_m bins, all terms >= 0) add at most (n_m + 2) U relative to the mel energy, 10 log10 turns that into
    DB_PER_REL (n_m + 2) U dB, and log10f and the product by 10 add about two ulps of the result."""
    n_terms = (mel_hi - mel_lo + 1).clamp_min(0).double().to(db64.device)
    return DB_PER_REL * (n_terms + 3) * U + 4 * U * db64.abs()


# ------------------------------------------------------------------------------------------------------------------
# CPU: the bounds reject the mistakes they stand for
# ------------------------------------------------------------------------------------------------------------------
def _tf32_rna(v):
    """fp32 -> tf32, round to nearest with ties away from zero (cvt.rna.tf32.f32; tf32_rna_host in lidfe_abi.cu)."""
    v = v.float().contiguous()
    u = ((v.view(torch.int32).long() & 0xFFFFFFFF) + 0x1000) & 0xFFFFE000
    r = torch.where(u >= 2 ** 31, u - 2 ** 32, u).to(torch.int32).view(torch.float32)
    return torch.where(torch.isfinite(v), r, v)


def _tf32_trunc(v):
    u = v.float().contiguous().view(torch.int32)
    return (u & ~0x1FFF).view(torch.float32)


def test_bounds_reject_emulated_kernel_mistakes():
    """The GEMM bound holds for the modelled kernel and fails for what a broken one would compute: one TF32 pass, a lost
    correction term (a lo image of zeros), a lost 32-tap block, the phases of a neighbouring tile -- on the 640- and
    2048-point DFT banks and the 44.1 kHz resampler bank.  The stft_mel_db bound holds for an fp32 evaluation and fails
    for a mel range shifted by one bin."""
    from speech_lid_b200 import tables
    x = O.synth_speechlike(48000, 11)[0]
    k, width = tables.sinc_resample_kernel(44100, 16000)
    cases = [(tables.windowed_dft_bank(640)[0], 320, 0), (tables.windowed_dft_bank(2048)[0], 1024, 0), (k, 441, width)]
    for bank, hop, left in cases:
        want, mag, acc, m3 = gemm_terms(x, bank, hop, left, passes=3)
        r = {p: gemm_ratio(gemm_terms(x, bank, hop, left, passes=p)[3], want, mag, acc) for p in (1, 2)}
        r3 = gemm_ratio(m3, want, mag, acc)
        print("bank %s: 3xTF32 %.3g, 2xTF32 %.3g, 1xTF32 %.3g of the bound" % (tuple(bank.shape), r3, r[2], r[1]))
        assert r3 <= 0.6, r3                 # the modelled kernel, rounding every accumulator update toward zero
        assert r[2] > 5 and r[1] > 10, r     # a dropped correction term, one TF32 pass
        holed = bank.clone()
        holed[:, 32:64] = 0                  # one 32-tap block lost (a pipeline item handed to the wrong set)
        assert gemm_ratio(gemm_terms(x, holed, hop, left, passes=3)[3], want, mag, acc) > 100
        swapped = bank.roll(1, 0)            # phases of a neighbouring tile / buffer
        assert gemm_ratio(gemm_terms(x, swapped, hop, left, passes=3)[3], want, mag, acc) > 100
    # stft_mel_db: an fp32 evaluation passes, a mel range shifted by one bin fails
    bank, hop = tables.windowed_dft_bank(640)[0], 320
    g = gemm_terms(x, bank, hop, 0, passes=3)[3]
    n_bins = 321
    melT = tables.htk_mel_banks(80, 640, 16000, 0.0, 8000.0)
    nz = melT != 0
    lo = torch.where(nz.any(1), nz.float().argmax(1), torch.zeros(80, dtype=torch.long))
    hi = torch.where(nz.any(1), n_bins - 1 - nz.flip(1).float().argmax(1), -torch.ones(80, dtype=torch.long))
    db64 = mel_db64(g, n_bins, melT)
    bound = mel_db_bound(db64, lo, hi)
    z = g[:, :2 * n_bins].reshape(-1, n_bins, 2)
    p32 = torch.addcmul(z[..., 1] * z[..., 1], z[..., 0], z[..., 0])
    db32 = 10.0 * torch.log10((p32 @ melT.T).clamp_min(1e-10))
    assert float(((db32.double() - db64).abs() / bound).max()) <= 1.0
    shifted = torch.zeros_like(melT)
    for m in range(80):
        if hi[m] >= lo[m]:
            cols = torch.arange(int(lo[m]) + 1, min(int(hi[m]) + 2, n_bins))
            shifted[m, cols] = melT[m, cols]
    db_s = 10.0 * torch.log10((p32.double() @ shifted.double().T).clamp_min(1e-10))
    assert float(((db_s - db64).abs() / bound).max()) > 100


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lid():
    import speech_lid_b200 as m
    return m


def _create(lid, row):
    old = os.environ.get("LIDFE_RESAMPLE_TC")
    if row["env"] is not None:
        os.environ["LIDFE_RESAMPLE_TC"] = row["env"]
    try:
        if row["kind"] == "rs":
            return lid.Resampler(row["orig"], row["new"])
        return lid.S3prlFBank(row["fbank_size"], row["n_fft"])
    finally:
        if old is None:
            os.environ.pop("LIDFE_RESAMPLE_TC", None)
        else:
            os.environ["LIDFE_RESAMPLE_TC"] = old


def _i64(v, dev):
    return torch.tensor(v, dtype=torch.int64, device=dev)


def _lidfe_resample(obj, packed, in_off, in_len, out, out_off, out_len):
    from speech_lid_b200 import _lib
    dev = packed.device
    t = [_i64(v, dev) for v in (in_off, in_len, out_off, out_len)]
    _lib.check(obj.lib.lidfe_resample(obj.handle, len(in_len), packed.data_ptr(), t[0].data_ptr(), t[1].data_ptr(),
                                      out.data_ptr(), t[2].data_ptr(), t[3].data_ptr(), max(out_len),
                                      torch.cuda.current_stream(dev).cuda_stream))
    torch.cuda.synchronize(dev)


def _check_kernels(fn, row, what):
    out, names = _cuda_kernels(fn)
    ran = _our_kernels(names)
    assert ran == set(row["kernels"]), (row["id"], what, sorted(ran), sorted(row["kernels"]))
    return out


def _walk_report(row, out_len, nw, max_out_len, sms):
    """Tiles per CTA of the launch (tensor-core rows); asserts some CTA takes >= 3 live tiles."""
    if row["tiling"] is None:
        return "-"
    live = tile_live(out_len, nw, row["tiling"][1], max_out_len)
    per = tiles_per_cta(live, sms)
    assert int(per.max()) >= 3, (row["id"], int(per.max()), int(live.sum()), live.numel())
    return int(per.max())


def _run_resampler(lid, row, dev, sms):
    rs = _create(lid, row)
    bank, hop, left = _geometry(row)
    nw = bank.shape[0]
    assert rs.kernel.shape == bank.shape and rs.width == left
    worst, per_cta = 0.0, "-"
    edge = [(_content(k, n, 9000 + i, False)[0], k) for i, (n, k) in enumerate(_edge_batch(row, hop))]
    for batch in ("edge", "walk"):
        if batch == "edge":
            wavs = [w.to(dev) for w, _ in edge]
            res = _check_kernels(lambda: rs.resample_list(wavs), row, batch)
        else:
            g = torch.Generator(device=dev).manual_seed(row["orig"] + row["new"])
            wavs = [torch.randn(n, generator=g, device=dev) for n in _walk_lengths(row, hop, (row["tiling"] or (0, 1))[1], sms)]
            res = rs.resample_list(wavs)
            out_len = [rs.out_len(w.numel()) for w in wavs]
            per_cta = _walk_report(row, out_len, nw, max(out_len), sms)
        for i, (w, y) in enumerate(zip(wavs, res)):
            want = O.truth64_resample(w, bank, left, row["orig"], row["new"])
            _, mag, acc, _ = gemm_terms(w, bank, hop, left)
            mag, acc = mag.reshape(-1)[:y.numel()], acc.reshape(-1)[:y.numel()]
            assert y.numel() == want.numel() == rs.out_len(w.numel()), (row["id"], batch, i)
            r = gemm_ratio(y, want, mag, acc)
            worst = max(worst, r)
            assert r <= 1.0, (row["id"], batch, i, w.numel(), r)
            if batch == "edge" and edge[i][1] == "zeros":
                assert torch.all(y == 0), (row["id"], i)
        if batch == "edge":
            edge_out = [y.clone() for y in res]
    # the tensor-core kernel agrees with the FP32 kernel of the same bank
    if TC in row["kernels"]:
        ref = _create(lid, dict(row, env="0"))
        wavs = [w.to(dev) for w, _ in edge]
        fp = _check_kernels(lambda: ref.resample_list(wavs), dict(row, kernels=frozenset([FP32])), "fp32 selector")
        scale = max(1.0, max(float(y.abs().max()) for y in fp if y.numel()))
        d = max(float((a - b).abs().max()) for a, b in zip(edge_out, fp) if a.numel())
        assert d <= 2e-6 * scale, (row["id"], d)
    # direct call: odd input offsets, outputs at gapped offsets (one not a multiple of 4), out_len cut short; the gaps
    # and everything past out_len keep the sentinel
    wavs = [w for w, _ in edge]
    packed, in_off = _pack(wavs, dev)
    full = [rs.out_len(w.numel()) for w in wavs]
    cut = [0, 1, full[2] // 3, 0, 5, full[5] - 1, 0, 1]
    out_len = [max(0, f - c) for f, c in zip(full, cut)]
    out_off, pos = [], 3
    for n in out_len:
        out_off.append(pos)
        pos += n + 5
    assert any(o % 4 for o in out_off)
    buf = torch.full((pos + 8,), SENTINEL, dtype=torch.int32, device=dev)
    _lidfe_resample(rs, packed, in_off, [w.numel() for w in wavs], buf.view(torch.float32), out_off, out_len)
    written = torch.zeros(buf.numel(), dtype=torch.bool, device=dev)
    for i, (o, n) in enumerate(zip(out_off, out_len)):
        got = buf[o:o + n].view(torch.float32)
        assert torch.equal(got, edge_out[i][:n]), (row["id"], "direct call", i)
        written[o:o + n] = True
    assert torch.all(buf[~written] == SENTINEL), (row["id"], "write outside out_off / out_len")
    return nw, per_cta, worst


def _s3_call(fb, wavs, dev, normalize):
    """S3prlFBank.forward_list's three launches on odd input offsets: (g, out rows, frames, first rows)."""
    from speech_lid_b200 import _lib
    packed, in_off = _pack(wavs, dev)
    n_in = [w.numel() for w in wavs]
    frames = [fb.num_frames(n) for n in n_in]
    g_off = [sum(frames[:i]) * fb.nw for i in range(len(wavs))]
    rows = [sum(frames[:i]) for i in range(len(wavs))]
    g = torch.full((sum(frames) * fb.nw,), float("nan"), dtype=torch.float32, device=dev)
    _lidfe_resample(fb, packed, in_off, n_in, g, g_off, [f * fb.nw for f in frames])
    out = torch.empty((sum(frames), fb.n_mels), dtype=torch.float32, device=dev)
    stats = torch.empty(2 * len(wavs), dtype=torch.float64, device=dev)
    go, fr, ro = _i64(g_off, dev), _i64(frames, dev), _i64(rows, dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(fb.lib.lidfe_stft_mel_db(g.data_ptr(), go.data_ptr(), fr.data_ptr(), len(wavs), max(frames), fb.nw,
                                        fb.melT.data_ptr(), fb.mel_lo.data_ptr(), fb.mel_hi.data_ptr(), fb.n_bins,
                                        fb.n_mels, 1e-10, out.data_ptr(), ro.data_ptr(), stats.data_ptr(),
                                        int(normalize), st))
    torch.cuda.synchronize(dev)
    return g, out, frames, rows


def _end_to_end(quads, what):
    """Pooled over a row's two batches, the median and the max of |gpu - truth| may not exceed 1.5x and 4x those of
    |model - truth|, model being the chain on the modelled GEMM (model_chain).  The fp32 oracle is no yardstick here:
    the tensor core rounds every accumulator update toward zero, and on coherent input (a periodic frame, a DFT bin
    near DC) those losses add up instead of cancelling, a bias of up to ~K/8 ulps of the bin that an fp32 FFT does not
    have; where a bin cancels (n_fft 4), the truncated lo operands of the 3 x TF32 split dominate.  The model carries
    both and puts the median error at 40x the oracle's at n_fft 640 and 120x at 2048 on speech-like input, its maximum
    at up to 18x on noise at n_fft 4: what the device shows.  Returns the device's median and max ratios to the model's
    and to the oracle's errors."""
    e = [torch.cat([(q[j].double() - q[3]).abs().reshape(-1) for q in quads]) for j in range(3)]
    med = [float(v.median()) for v in e]
    mx = [float(v.max()) for v in e]
    assert med[0] <= 1.5 * med[1] and mx[0] <= 4.0 * mx[1], (what, "median gpu / model", med[0], med[1],
                                                           "max gpu / model", mx[0], mx[1])
    r = lambda a, b: a / b if b else (0.0 if a == 0 else float("inf"))     # noqa: E731
    return r(med[0], med[1]), r(mx[0], mx[1]), r(med[0], med[2]), r(mx[0], mx[2])


def _run_s3prl(lid, row, dev, sms):
    fb = _create(lid, row)
    bank, hop, left = _geometry(row)
    nw, n_fft, n_bins, n_mels = fb.nw, row["n_fft"], fb.n_bins, fb.n_mels
    assert bank.shape == (nw, n_fft)
    lo, hi = fb.mel_lo.long(), fb.mel_hi.long()
    worst, per_cta, e2e = 0.0, "-", (0.0,) * 4
    pairs_raw, pairs_norm = [], []        # pooled over both batches: the edge batch alone holds a few hundred values
    for batch in ("edge", "walk"):
        if batch == "edge":
            spec = _edge_batch(row, hop)
            wavs = [_content(k, n, 7000 + i, False)[0] for i, (n, k) in enumerate(spec)]
            kinds = [k for _, k in spec]
            dwavs = [w.to(dev) for w in wavs]
            ref_norm = _check_kernels(lambda: fb.forward_list(dwavs), row, batch)
            ref_raw = fb.forward_list(dwavs, normalize=False)
        else:
            g_ = torch.Generator(device=dev).manual_seed(n_fft + row["fbank_size"])
            dwavs = [torch.randn(n, generator=g_, device=dev) for n in _walk_lengths(row, hop, row["tiling"][1], sms)]
            wavs = [w.cpu() for w in dwavs]
            kinds = ["noise"] * len(wavs)
            ref_raw = None
        g, raw, frames, rows = _s3_call(fb, dwavs, dev, False)
        _, norm, _, _ = _s3_call(fb, dwavs, dev, True)
        if batch == "walk":
            per_cta = _walk_report(row, [f * nw for f in frames], nw, max(frames) * nw, sms)
        for i, (w, kind) in enumerate(zip(dwavs, kinds)):
            T = frames[i]
            what = (row["id"], batch, i, kind, w.numel())
            # 1. GEMM rows against float64 frames x the same fp32 bank; the zero rows of the bank give exact zeros
            gi = g[sum(frames[:i]) * nw:(sum(frames[:i]) + T) * nw].view(T, nw)
            want, mag, acc, model = (v[:T] for v in gemm_terms(w, bank, hop, left, passes=3))
            r = gemm_ratio(gi, want, mag, acc)
            worst = max(worst, r)
            assert r <= 1.0, what + (r,)
            assert torch.all(gi[:, 2 * n_bins:] == 0), what
            # 2. power -> mel -> dB of the device's own GEMM rows
            db = raw[rows[i]:rows[i] + T]
            db64 = mel_db64(gi, n_bins, fb.melT)
            excess = float(((db.double() - db64).abs() / mel_db_bound(db64, lo, hi)).max())
            assert excess <= 1.0, what + ("stft_mel_db", excess)
            empty = (hi < lo).to(dev)
            assert torch.all(db[:, empty] == -100.0), what             # filters without a bin: exactly the floor
            # 3. scalar normalisation against float64 statistics of the device's own dB rows
            nz = norm[rows[i]:rows[i] + T]
            n = T * n_mels
            if n == 1:
                assert torch.isnan(nz).all(), what                     # torch.std of one value
            else:
                d64 = db.double()
                std, mean = torch.std_mean(d64)
                want_n = (d64 - mean) / (std + 1e-9)
                err = (nz.double() - want_n).abs()
                assert float((err / (5 * U * (want_n.abs() + 1))).max()) <= 1.0, what + ("scalar_norm", float(err.max()))
            if kind == "zeros":
                assert torch.all(db == -100.0) and torch.all(nz == 0.0), what
                continue
            # 4. end to end against the fp64 reference, pooled below
            tr = O.truth64_s3prl_fbank(w, row["fbank_size"], n_fft, False)
            tn = O.truth64_s3prl_fbank(w, row["fbank_size"], n_fft, True)
            orr = O.s3prl_fbank(wavs[i], row["fbank_size"], n_fft, False).T.to(dev)
            onn = O.s3prl_fbank(wavs[i], row["fbank_size"], n_fft, True).T.to(dev)
            mr, mn = model_chain(model, n_bins, fb.melT)
            assert tr.shape == db.shape == orr.shape == mr.shape, what
            pairs_raw.append((db, mr, orr, tr))
            if n > 1:
                pairs_norm.append((nz, mn, onn, tn))
        if ref_raw is not None:
            # the direct calls on odd input offsets give forward_list's bits
            for i, T in enumerate(frames):
                assert torch.equal(ref_raw[i], raw[rows[i]:rows[i] + T]), (row["id"], i)
                assert torch.allclose(ref_norm[i], norm[rows[i]:rows[i] + T], rtol=1e-6, atol=1e-6, equal_nan=True)
    for pairs, what in ((pairs_raw, "dB"), (pairs_norm, "normalised")):
        e2e = tuple(max(a, b) for a, b in zip(e2e, _end_to_end(pairs, (row["id"], what))))
    return nw, per_cta, worst, e2e


@gpu
@pytest.mark.parametrize("row", ROWS, ids=[r["id"] for r in ROWS])
def test_gemm_route(lid, row):
    dev = torch.device("cuda", torch.cuda.current_device())
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    if row["kind"] == "rs":
        nw, per_cta, worst = _run_resampler(lid, row, dev, sms)
        extra = ""
    else:
        nw, per_cta, worst, e2e = _run_s3prl(lid, row, dev, sms)
        extra = (", |gpu - truth64| over |model - truth64|: median %.2f, max %.2f; over |oracle32 - truth64|: "
                 "median %.2f, max %.2f" % e2e)
    kernel = TC if TC in row["kernels"] else FP32
    t = row["tiling"] or ("-",) * 4
    print("%s: %s nw %d N %s tiles %s KB %s stages %s, max tiles/CTA %s, worst error/bound %.3g%s"
          % (row["id"], kernel, nw, t[0], t[1], t[2], t[3], per_cta, worst, extra))


@gpu
def test_s3prl_silence_and_single_value(lid):
    """Silence: exactly -100 dB and exactly 0 after normalisation; one value (fbank_size 1, one frame): NaN, as torch.std."""
    dev = torch.device("cuda", torch.cuda.current_device())
    fb = lid.S3prlFBank(80, 640)
    for n in (640, 641, 6400):
        z = fb.forward_list([torch.zeros(n, device=dev)], normalize=False)[0]
        assert torch.all(z == -100.0)
        assert torch.all(fb.forward_list([torch.zeros(n, device=dev)])[0] == 0.0)
    one = lid.S3prlFBank(1, 640).forward_list([torch.randn(640, device=dev)])[0]
    assert one.shape == (1, 1) and bool(torch.isnan(one).all())
