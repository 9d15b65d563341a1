// lidfe_mfcc_mma.cuh -- the DCT-II + lifter of the two-kernel MFCC path (row A5; ta: compliance/kaldi.py:648-666, 669-813) on
// the tensor cores.
//
// The in-kernel DCT epilogue of fbank_kernel re-reads the n_mels x n_ceps matrix from shared memory for every frame pair
// (+65 % shared-memory wavefronts on a kernel that is bound by exactly that pipe); when no statistics are needed (cmvn
// none / global apply) the fbank kernel writes the log-mels to a tile-blocked workspace (FbankParams::ws_blocked) and this
// kernel finishes the job.  [rows x n_mels] . [n_mels x n_ceps] is 6.4 kflop per frame: as FP32 FMAs (a register-tiled
// kernel, measured, then removed; see git history) it cost 47 us per 512 x 4 s against an HBM floor of 15 us (65 MB of
// log-mels in, 33 MB of cepstra out).  Here the product runs as 3xTF32
// (hi = tf32(v), lo = v - hi; D += A_lo B_hi + A_hi B_lo + A_hi B_hi with fp32 accumulation: ~21 mantissa bits per
// product, the decomposition of resample_tc_kernel) on mma.sync.m16n8k8 -- 150 MMAs per 16-frame tile:
//   * the tile-blocked log-mel workspace [tile][mel / 4][16 frames][4] IS the A-fragment order: a0 of the 32 lanes for
//     k-step ks is the 128 contiguous bytes at (2 ks) * 256, a1 the next 128, a2 / a3 the 256 bytes after that;
//   * every warp owns a contiguous range of tiles; a tile (16 frames, 5 KB) arrives by ONE TMA bulk copy
//     (cp.async.bulk + mbarrier) into the warp's double buffer while the previous one is multiplied; the first copy is
//     issued before the CTA sets up its tables;
//   * the DCT matrix is split once per CTA into hi / lo images laid out in B-fragment order (one conflict-free LDS.64
//     per lane, k-step and 8-column block);
//   * the three partial products are three SWEEPS over the column-block accumulators, so that consecutive MMAs are
//     independent (a dependent chain of three per accumulator ran at the MMA latency: slower than the FP32 kernel).
// Epilogue: lifter, global CMVN, SpecAugment zero-fill, stores of two adjacent cepstra per lane.
// MEASURED (cfg3, 512 x 4 s, one B200): 35-37 us against 47 us for the FP32 kernel (cfg3 step 148 -> 136 us).  ncu: the
// tensor pipe is 49 % busy -- the legacy mma.sync TF32 path retires an m16n8k8 in 2.8 cycles per SM, so the 1.92 M MMAs
// of a launch are 18.5 us by themselves; 8 warps per SM with two tiles per pass were slower (47 us), 16 warps with one
// tile per pass are what is kept.  The HBM floor (15 us) would need the tcgen05 path (resample_tc_kernel's machinery
// plus a K-major workspace), not built.
// Scope: n_mels % 4 == 0, n_ceps <= 40 (when n_mels % 8 == 4 the last k-step has half its mel bins, the other half is
// zero on both sides).
#pragma once
#include "lidfe_kernels.cuh"

namespace lidfe {

constexpr int kDctMaxCeps = 40;                 // n_ceps <= 40 takes the two-kernel path

struct DctParams {
  const float* logmel;      // workspace [n_tiles][n_mels / 4][16][4]
  float* out;
  long long out_ld;
  const Tile* tiles;
  int n_tiles;
  int n_mels, n_ceps;       // n_mels % 4 == 0
  const float* dct;         // [n_mels][n_ceps] device copy
  const float* lifter;      // [n_ceps]
  const int* masks;
  int n_masks;
  int mode;                 // 0 none, 2 global apply
  const double* stats_in;   // [2*n_ceps+1] (mode 2)
};

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

constexpr int kMmTM = 1;                        // tiles per pass and warp
constexpr int kMmThreads = 256;
constexpr int kMmWarps = kMmThreads / 32;
constexpr int kMmMaxKS = kMaxMels / 8;          // k-steps (8 mel bins each)
constexpr int kMmMaxNT = kDctMaxCeps / 8;       // 8-column blocks of cepstra
constexpr int kMmPairBytes = kMmTM * kTileFrames * kMaxMels * 4;  // kMmTM tiles of 16 x 80 floats (5120 B each)
// dynamic shared memory: B images hi | lo  [KS][NT][32 lanes][2] floats each, lifter[40], norm[40] float2,
// per warp: mbarriers[2] (16 B) + 2 tile buffers
constexpr int kMmOffLift = 2 * kMmMaxKS * kMmMaxNT * 64 * 4;                 // 25600
constexpr int kMmOffNorm = kMmOffLift + kDctMaxCeps * 4;
constexpr int kMmOffBar = kMmOffNorm + kDctMaxCeps * 8;                      // 16 B per warp
constexpr int kMmOffBuf = (kMmOffBar + kMmWarps * 16 + 127) / 128 * 128;
constexpr int kMmSmemBytes = kMmOffBuf + kMmWarps * 2 * kMmPairBytes;        // ~108 KB -> 2 CTAs per SM

__global__ void __launch_bounds__(kMmThreads, 2) mfcc_dct_mma_kernel(const __grid_constant__ DctParams P) {
  extern __shared__ __align__(128) unsigned char msm[];
  float* const s_bhi = reinterpret_cast<float*>(msm);
  float* const s_blo = s_bhi + kMmMaxKS * kMmMaxNT * 64;
  float* const s_lift = reinterpret_cast<float*>(msm + kMmOffLift);
  float2* const s_norm = reinterpret_cast<float2*>(msm + kMmOffNorm);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, c = lane & 3;
  uint64_t* const bars = reinterpret_cast<uint64_t*>(msm + kMmOffBar + warp * 16);
  unsigned char* const bufs = msm + kMmOffBuf + warp * 2 * kMmPairBytes;

  const int nm = P.n_mels, nc = P.n_ceps;
  const int KS = (nm + 7) >> 3, NT = (nc + 7) >> 3;
  const int tile_bytes = kTileFrames * nm * 4;

  // ---- this warp's contiguous range of tiles; its first copy goes out before anything else, so that it flies under the
  //      set-up of the B images ---------------------------------------------------------------------------------------
  const long long gtid = static_cast<long long>(blockIdx.x) * kMmThreads + tid;
  const long long nthreads = static_cast<long long>(gridDim.x) * kMmThreads;
  const bool vec_out = (P.out_ld % 2 == 0) && ((reinterpret_cast<uintptr_t>(P.out) & 7) == 0);
  const long long gw = gtid >> 5, nwarps = nthreads >> 5;
  const long long base = P.n_tiles / nwarps, rem = P.n_tiles - base * nwarps;
  long long t = gw * base + (gw < rem ? gw : rem);
  const long long t_end = t + base + (gw < rem ? 1 : 0);

  auto issue = [&](long long t0, int which) {        // lane 0: kMmTM tiles starting at tile t0 -> buffer `which`
    const int n = (t0 + kMmTM <= t_end) ? kMmTM : static_cast<int>(t_end - t0);
    const uint32_t bytes = static_cast<uint32_t>(n * tile_bytes);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(bars + which, bytes);
    tma_bulk_g2s(bufs + which * kMmPairBytes, P.logmel + t0 * (kTileFrames * nm), bytes, bars + which, l2_evict_first_policy());
  };
  if (lane == 0) {
    mbar_init(bars, 1);
    mbar_init(bars + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (t < t_end) issue(t, 0);
  }

  // ---- B images: element (k, n) of the DCT matrix for lane (g, c): b0 = (8 ks + c, 8 nt + g), b1 = (8 ks + c + 4, 8 nt + g)
  for (int e = tid; e < KS * kMmMaxNT * 64; e += kMmThreads) {      // (column blocks beyond n_ceps, rows beyond n_mels are zeros)
    const int which = e & 1, ln = (e >> 1) & 31, blk = e >> 6;
    const int ks = blk / kMmMaxNT, nt = blk - ks * kMmMaxNT;
    const int k = 8 * ks + (ln & 3) + 4 * which, n = 8 * nt + (ln >> 2);
    const float v = (n < nc && k < nm) ? __ldg(P.dct + k * nc + n) : 0.f;
    uint32_t hi, lo;
    split_tf32(v, hi, lo);
    s_bhi[e] = __uint_as_float(hi);
    s_blo[e] = __uint_as_float(lo);
  }
  if (tid < kDctMaxCeps) {
    s_lift[tid] = tid < nc ? P.lifter[tid] : 0.f;
    float mean = 0.f, inv = 1.f;
    if (P.mode == 2 && tid < nc) {
      const double n = P.stats_in[2 * nc];
      const double mu = P.stats_in[tid] / n;
      double var = (P.stats_in[nc + tid] - P.stats_in[tid] * mu) / (n - 1.0);
      var = var > 0.0 ? var : 0.0;
      mean = static_cast<float>(mu);
      inv = static_cast<float>(1.0 / (sqrt(var) + 1e-9));
    }
    s_norm[tid] = make_float2(mean, inv);
  }
  __syncthreads();

  uint32_t ph0 = 0u, ph1 = 0u;
  int cur = 0;
  for (; t < t_end; t += kMmTM) {
    const int n_here = (t + kMmTM <= t_end) ? kMmTM : static_cast<int>(t_end - t);
    if (lane == 0 && t + kMmTM < t_end) issue(t + kMmTM, cur ^ 1);      // the other buffer was read to the end a pass ago (syncwarp below)
    Tile tls[kMmTM];            // descriptors of the pass, asked for before the wait: their latency hides under the MMAs
#pragma unroll
    for (int i = 0; i < kMmTM; ++i) tls[i] = P.tiles[(t + i < t_end) ? t + i : t];
    mbar_wait(bars + cur, cur ? ph1 : ph0);
    if (cur) ph1 ^= 1u; else ph0 ^= 1u;
    const float* A = reinterpret_cast<const float*>(bufs + cur * kMmPairBytes);

    float acc[kMmTM][kMmMaxNT][4];
#pragma unroll
    for (int i = 0; i < kMmTM; ++i)
#pragma unroll
      for (int nt = 0; nt < kMmMaxNT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[i][nt][e] = 0.f;

#pragma unroll 2
    for (int ks = 0; ks < KS; ++ks) {
      uint32_t ahi[kMmTM][4], alo[kMmTM][4];
      // mel bins 8 ks + 4 .. 8 ks + 7 lie past the tile when n_mels % 8 == 4 and this is the last k-step: a2 / a3 must be
      // zeros, not the stale bytes behind the tile (a NaN there times the zero rows of B is still NaN)
      const bool quad2 = 8 * ks + 4 < nm;
#pragma unroll
      for (int i = 0; i < kMmTM; ++i) {
        const float* a = A + i * (kTileFrames * nm) + ks * 128 + lane;
        split_tf32(a[0], ahi[i][0], alo[i][0]);
        split_tf32(a[32], ahi[i][1], alo[i][1]);
        split_tf32(quad2 ? a[64] : 0.f, ahi[i][2], alo[i][2]);
        split_tf32(quad2 ? a[96] : 0.f, ahi[i][3], alo[i][3]);
      }
      // B fragments of the k-step for every column block, then the three partial products as three SWEEPS over the
      // (tile, column block) accumulators: consecutive MMAs are independent (a dependent chain of three per accumulator
      // issued back to back ran at the MMA latency: 165 us per cfg3 step instead of 148 for the FP32 kernel)
      uint32_t bh[kMmMaxNT][2], bl[kMmMaxNT][2];
#pragma unroll
      for (int nt = 0; nt < kMmMaxNT; ++nt) {
        const float2 vh = *reinterpret_cast<const float2*>(s_bhi + (ks * kMmMaxNT + nt) * 64 + lane * 2);
        const float2 vl = *reinterpret_cast<const float2*>(s_blo + (ks * kMmMaxNT + nt) * 64 + lane * 2);
        bh[nt][0] = __float_as_uint(vh.x); bh[nt][1] = __float_as_uint(vh.y);
        bl[nt][0] = __float_as_uint(vl.x); bl[nt][1] = __float_as_uint(vl.y);
      }
      // (no conditions between the MMAs: an absent second tile multiplies stale bytes into accumulators nobody stores,
      // column blocks beyond n_ceps multiply zeros)
#pragma unroll
      for (int term = 0; term < 3; ++term) {
#pragma unroll
        for (int nt = 0; nt < kMmMaxNT; ++nt) {
#pragma unroll
          for (int i = 0; i < kMmTM; ++i) {
            if (term == 0) mma_tf32(acc[i][nt], alo[i], bh[nt][0], bh[nt][1]);
            else if (term == 1) mma_tf32(acc[i][nt], ahi[i], bl[nt][0], bl[nt][1]);
            else mma_tf32(acc[i][nt], ahi[i], bh[nt][0], bh[nt][1]);
          }
        }
      }
    }
    __syncwarp();        // every lane has read the tile: the buffer may be refilled by the copy issued next pass
    cur ^= 1;

    // ---- epilogue: lifter, global CMVN, SpecAugment zero-fill, store (lane holds frames g, g + 8 x cepstra 8 nt + 2 c, + 1)
#pragma unroll
    for (int i = 0; i < kMmTM; ++i) {
      if (i >= n_here) continue;
      const Tile tl = tls[i];
      const int* mk = P.masks + static_cast<long long>(tl.utt) * P.n_masks * 4;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int fr = g + 8 * h;
        if (fr >= tl.nframes) continue;
        const int tf = tl.t0 + fr;
        bool row_masked = false;
        for (int qm = 0; qm < P.n_masks; ++qm) row_masked |= (tf >= mk[4 * qm] && tf < mk[4 * qm + 1]);
        float* o = P.out + (tl.out_row + fr) * P.out_ld;
#pragma unroll
        for (int nt = 0; nt < kMmMaxNT; ++nt) {
          if (nt >= NT) continue;
          const int j0 = 8 * nt + 2 * c;
          float x[2] = {acc[i][nt][2 * h], acc[i][nt][2 * h + 1]};
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int j = j0 + e;
            float v = __fmul_rn(x[e], s_lift[j < kDctMaxCeps ? j : 0]);
            if (P.mode == 2) v = (v - s_norm[j < kDctMaxCeps ? j : 0].x) * s_norm[j < kDctMaxCeps ? j : 0].y;
            bool z = row_masked;
            for (int qm = 0; qm < P.n_masks; ++qm) z |= (j >= mk[4 * qm + 2] && j < mk[4 * qm + 3]);
            x[e] = z ? 0.f : v;
          }
          if (vec_out && j0 + 1 < nc) *reinterpret_cast<float2*>(o + j0) = make_float2(x[0], x[1]);
          else {
            if (j0 < nc) o[j0] = x[0];
            if (j0 + 1 < nc) o[j0 + 1] = x[1];
          }
        }
      }
    }
  }

  // zero-fill tiles (pad_sequence's zeros): 4 threads per tile
  for (long long q = gtid; q < static_cast<long long>(P.n_tiles) * 4; q += nthreads) {
    const Tile tl = P.tiles[q >> 2];
    if (tl.nframes != 0) continue;
    for (int r = static_cast<int>(q & 3); r < tl.aux; r += 4) {
      float* o = P.out + (tl.out_row + r) * P.out_ld;
      for (int j = 0; j < nc; ++j) o[j] = 0.f;
    }
  }
}

}  // namespace lidfe
