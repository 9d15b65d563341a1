// lidfe_abi.cu -- C ABI (include/lidfe.h) over the sm_100a kernels in lidfe_kernels.cuh.
// Host side only builds constant tables / the per-batch tile table and launches kernels; there is no
// CPU compute path.
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "../../include/lidfe.h"
#include "lidfe_kernels.cuh"
#include "lidfe_fbank_warp.cuh"
#include "lidfe_resample_tc.cuh"
#include "lidfe_stft_fbank.cuh"
#include "lidfe_fbank_precise.cuh"
#include "lidfe_mfcc_mma.cuh"

using namespace lidfe;

// One pooled allocation behind a plan: a device block, its pinned host mirror (the staging buffer of the single
// table upload) and the event that marks the last device work that touched them.  Blocks live in the handle's pool:
// lidfe_plan_destroy hands them back, lidfe_plan_create_async re-uses the first one that is large enough, so ragged
// batches (a new length signature every step, ref: lid/raw_datasets.py:345-365) allocate nothing in steady state.
//
// Layout (sized by CAPACITY, so the at-rest state survives re-use with another batch size):
//   workspace  sched[2] int | utt_max[2][Bc] u32 (0) | utt_min[2][Bc] u32 (~0) | utt_stats[2][Bc][2][n_out] f64 (0) |
//              utt_wnorm[Bc] float2                                ([2] = launch parity, see FbankParams::utt_stats)
//   tables     frames[Bc] i64 | out_rows[Bc] i64 | offsets[Bc] i64 | lengths[Bc] i64 | first_tile[Bc] i64 |
//              spans[Sc] | w_first[W + 1] int | warp spans[Wc] | tiles[Tc] (MFCC two-kernel path only)
struct PlanBlock {
  unsigned char* d_base;
  unsigned char* h_tables;      // pinned mirror of the tables section
  size_t ws_bytes, tab_bytes;
  int Bc;
  long long Sc, Tc, Wc;         // capacities: spans, tiles, warp spans
  cudaEvent_t ev;               // last use on the device (kernels or the upload)
  float* d_logmel;              // tile-blocked log-mel workspace of the two-kernel MFCC path (grown on demand)
  long long logmel_tiles;
};

// Created value-initialised (new lidfe_ctx()): every scalar member starts at zero.
struct lidfe_ctx {
  lidfe_config cfg;
  int device;
  int num_sms;
  int n_out;
  int band_taps[kBands];
  int std_mel;    // kernel variant: 1 = Kaldi-80 bank + DC removal + pre-emphasis 1.0, 2 = HTK-80 bank + window-only
                  // framing (both with the mel loop fully unrolled), 0 = generic (runtime loops and switches)
  // device tables
  unsigned char* d_blob;   // window | tw1 | tw2 | mel_k0 | mel_w | dct | lifter, laid out like the kernel's shared memory
  int blob_bytes;
  int blob_bytes_fbank;    // prefix without dct / lifter (the fbank-only kernel variant of the two-kernel MFCC path)
  int dct_off, lifter_off; // byte offsets of those sections inside the blob
  size_t smem_bytes_fbank;
  size_t smem_bytes;
  int grid_cap;   // resident CTAs of the fbank kernel on this device
  // warp-autonomous kernel (lidfe_fbank_warp.cuh); route_for decides when it runs
  bool warp_off;      // LIDFE_WARP_KERNEL=0 at creation
  int w_grid;         // resident CTAs of that kernel (0 when the handle cannot use it)
  int w_tab_bytes;    // shared-memory bytes in front of the per-warp areas
  size_t w_smem;      // dynamic shared memory per CTA
  std::vector<PlanBlock*> pool;       // free blocks
  std::mutex pool_mu;
  long long blocks_allocated;         // device/pinned block allocations made for plans so far (lidfe_pool_stats)
  int live_plans;                     // plans that still point at this handle (guarded by pool_mu)
  bool destroyed;                     // lidfe_destroy was called while plans were alive: the last plan frees the handle
  // optional per-launch timing of the fbank kernel (bench.py's roofline leg)
  std::vector<cudaEvent_t> prof_events;   // empty outside lidfe_profile_begin / lidfe_profile_end
  int prof_used;
  int prof_stride;   // bracket every prof_stride-th featurize call (event records between kernels cost a few us)
  int prof_calls;
  // precise mode (lidfe_set_precision, lidfe_fbank_precise.cuh): fp64 arithmetic on the reference's fp32 tables
  int precise;
  int k0_off, melw_off, total_taps;   // the segment-form mel plan inside the blob (the precise kernel reads it from there)
};

struct lidfe_plan_s {
  lidfe_ctx* ctx;
  int B;
  long long total_frames;
  long long n_tiles;
  long long n_spans;
  std::vector<long long> frames;
  PlanBlock* blk;
  // views into blk->d_base
  int* d_sched;
  unsigned* d_utt_max;
  unsigned* d_utt_min;
  double* d_utt_stats;
  float2* d_utt_wnorm;
  int parity;             // per-utterance launches on this plan so far, mod 2 (host-side toggle)
  long long* d_frames;    // [B]
  long long* d_out_rows;  // [B]
  long long* d_offsets;   // [B]
  long long* d_lengths;   // [B]
  long long* d_utt_first_tile;   // [B]
  Span* d_spans;
  Span* d_wspans;         // warp spans (NULL unless plan_can_warp)
  long long n_wspans;
  int n_wstatic;          // spans [0, n_wstatic) are the warps' static runs, the rest is the pool
  int* d_w_first;         // [W + 1] first static span of every warp
  bool all_aligned;       // every utterance starts on a 16-byte boundary (TMA-eligible)
  Tile* d_tiles;          // MFCC two-kernel path (handle_has_dct_path), else NULL
  long long max_frames;
  long long max_row;      // rows of the output matrix this plan touches
};

static std::atomic<long long> g_launches{0};

#define CU_TRY(expr)                      \
  do {                                    \
    cudaError_t e__ = (expr);             \
    if (e__ != cudaSuccess) {             \
      cudaGetLastError();                 \
      return static_cast<int>(e__);       \
    }                                     \
  } while (0)

template <typename T>
static cudaError_t upload(T** dst, const T* src, size_t n) {
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(dst), n * sizeof(T));
  if (e != cudaSuccess) return e;
  return cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice);
}

typedef void (*fbank_fn)(const FbankParams);
// stats: 0 = none, 1 = sums (per-utterance / global CMVN), 2 = extrema (AmplitudeToDB top_db)
template <typename TIn>
static fbank_fn pick_warp_kernel_t(int std_mel, int stats) {
  if (std_mel == 2) return stats == 2 ? fbank_warp_kernel<TIn, 2, 2> : stats == 1 ? fbank_warp_kernel<TIn, 2, 1> : fbank_warp_kernel<TIn, 2, 0>;
  if (std_mel == 1) return stats == 1 ? fbank_warp_kernel<TIn, 1, 1> : fbank_warp_kernel<TIn, 1, 0>;
  return stats == 1 ? fbank_warp_kernel<TIn, 0, 1> : fbank_warp_kernel<TIn, 0, 0>;
}
static fbank_fn pick_warp_kernel(int in_dtype, int std_mel, int stats) {
  return in_dtype == LIDFE_IN_I16 ? pick_warp_kernel_t<short>(std_mel, stats) : pick_warp_kernel_t<float>(std_mel, stats);
}
template <typename TIn>
static fbank_fn pick_kernel_t(bool mfcc, int std_mel) {
  if (mfcc) return std_mel == 1 ? fbank_kernel<TIn, true, 1> : std_mel == 2 ? fbank_kernel<TIn, true, 2> : fbank_kernel<TIn, true, 0>;
  return std_mel == 1 ? fbank_kernel<TIn, false, 1> : std_mel == 2 ? fbank_kernel<TIn, false, 2> : fbank_kernel<TIn, false, 0>;
}
static fbank_fn pick_kernel(int in_dtype, bool mfcc, int std_mel) {
  return in_dtype == LIDFE_IN_I16 ? pick_kernel_t<short>(mfcc, std_mel) : pick_kernel_t<float>(mfcc, std_mel);
}
static size_t smem_for(const lidfe_config& c, int total_taps) {
  const bool mf = c.n_ceps > 0;
  const size_t base = (c.in_dtype == LIDFE_IN_I16)
                          ? (mf ? SmemLayout<short, true>::off_melw : SmemLayout<short, false>::off_melw)
                          : (mf ? SmemLayout<float, true>::off_melw : SmemLayout<float, false>::off_melw);
  size_t extra = static_cast<size_t>(total_taps) * 32;   // (wa, wb) per step and lane
  if (c.n_ceps > 0) extra += ((static_cast<size_t>(c.n_mels) * c.n_ceps + 3) & ~static_cast<size_t>(3)) + ((c.n_ceps + 3) & ~3);
  return base + extra * sizeof(float);
}

// ------------------------------------------------------------------------------------------------------------------
// Routing: which kernels serve a featurize call.  route_for holds the rule; lidfe_create sets up, and
// lidfe_plan_create_async builds the work lists for, whatever its predicates allow.
// ------------------------------------------------------------------------------------------------------------------
// fbank_warp_kernel's scope (lidfe_fbank_warp.cuh), as far as the configuration decides it: no in-kernel dither, and
// KALDI framing with a generic or the Kaldi-80 bank, or the reference's default branch as a whole (CENTER framing,
// HTK-80 bank, window-only framing, fbank output) with a pad of a multiple of 16 bytes of input (4 float or 8 int16
// samples), so that the interior quads of a 16-byte aligned utterance stay on 16-byte boundaries
static bool handle_can_warp(const lidfe_ctx* h) {
  const lidfe_config& c = h->cfg;
  const int in_elt = (c.in_dtype == LIDFE_IN_I16) ? 2 : 4;
  const bool kaldi = c.framing == LIDFE_FRAMING_KALDI && h->std_mel != 2;
  const bool center = c.framing == LIDFE_FRAMING_CENTER && h->std_mel == 2 && c.n_ceps == 0 && (c.pad * in_elt) % 16 == 0;
  return c.dither == 0.f && (kaldi || center) && !h->warp_off;
}
// ... and every utterance of the plan starts on a 16-byte boundary (the kernel stages quads with bulk copies only)
static bool plan_can_warp(const lidfe_ctx* h, bool aligned) { return aligned && handle_can_warp(h); }
// MFCC without statistics may run as fbank into a log-mel workspace, then mfcc_dct_mma_kernel (its table: n_mels % 4 == 0)
static bool handle_has_dct_path(const lidfe_ctx* h) {
  return h->cfg.n_ceps > 0 && h->cfg.n_ceps <= kDctMaxCeps && h->cfg.n_mels % 4 == 0;
}

enum FbankKind { kFbPrecise, kFbWarp, kFbCta };
// the cmvn_apply_kernel pass after the feature kernels: none, per-utterance normalisation or the top_db clamp (the
// statistics of this launch's parity), global statistics, masks only
enum ApplyPass { kApplyNone, kApplyUtt, kApplyTopDb, kApplyGlobal, kApplyMasks };
struct Route {
  FbankKind fbank;
  fbank_fn fn;        // the warp or CTA instantiation (precise: launch_precise picks it)
  bool dct;           // fbank into the tile-blocked log-mel workspace, then mfcc_dct_mma_kernel into the output
  ApplyPass apply;
};

static Route route_for(const lidfe_ctx* h, const lidfe_plan_s* p, int mode, bool raw, bool masks) {
  Route r = {kFbCta, nullptr, false, kApplyNone};
  if (mode == LIDFE_CMVN_PER_UTT) r.apply = kApplyUtt;
  if (mode == LIDFE_POST_TOPDB) r.apply = kApplyTopDb;
  if (h->precise) {   // fbank_precise_kernel takes statistics but leaves global CMVN and masks to the apply pass
    r.fbank = kFbPrecise;
    if (mode == LIDFE_CMVN_APPLY_GLOBAL) r.apply = kApplyGlobal;
    if (mode == LIDFE_CMVN_NONE && masks) r.apply = kApplyMasks;
    return r;
  }
  const lidfe_config& c = h->cfg;
  r.dct = handle_has_dct_path(h) && (mode == LIDFE_CMVN_NONE || mode == LIDFE_CMVN_APPLY_GLOBAL);
  // the warp kernel has no fused normalize_wav load, no in-kernel DCT and takes extrema only in the std_mel 2 variant
  const bool warp = !raw && plan_can_warp(h, p->all_aligned) && (c.n_ceps == 0 || r.dct) &&
                    (mode != LIDFE_POST_TOPDB || h->std_mel == 2);
  if (warp) {
    const int stats = r.dct ? 0 : (mode == LIDFE_CMVN_PER_UTT || mode == LIDFE_CMVN_ACCUM_GLOBAL) ? 1 : mode == LIDFE_POST_TOPDB ? 2 : 0;
    r.fbank = kFbWarp;
    r.fn = pick_warp_kernel(c.in_dtype, h->std_mel, stats);
  } else {
    r.fn = pick_kernel(c.in_dtype, c.n_ceps > 0 && !r.dct, h->std_mel);
  }
  return r;
}

// ------------------------------------------------------------------------------------------------------------------
// Mel plan.  The banks the reference uses (Kaldi and HTK triangles, ta: compliance/kaldi.py:436-511,
// functional/functional.py melscale_fbanks) overlap only with their neighbours: the FFT bins between the centres of
// filters j and j+1 ("segment j+1") carry the down-slope of filter j and the up-slope of filter j+1 and nothing else.
// So instead of letting every filter gather its whole support (every power bin read twice), slot j = lane j % 16 of
// band j / 16 walks segment j+1 once with TWO weights per bin -- wa into its own filter j, wb into a carry that the
// next lane adds to filter j+1 (one shuffle per band).  Segment 0 (bins below the first centre) is prepended to slot
// 0's run with wb = 0.  257 power bins are read per frame instead of 501 (+ padding), in ~22 steps instead of 41.
//
// Tap placement.  At step i the 16 lanes of a half-warp read the power pairs P[start_t + i] (8 bytes each).  Two lanes
// collide in shared memory when their starts differ but are congruent mod 16 (same bank pair, different address).  A
// run of len bins can start anywhere in [first + len - T, first] when the band runs T >= len steps (leading / trailing
// weights are zero), so for each band we look for the smallest T for which the lanes can be matched to 16 distinct
// residue classes (an exact bipartite matching), or, failing that, share classes between lanes that read the very same
// address (a bounded search: a lane may evict a class if every evicted lane can be re-seated, depth <= 3).
// ------------------------------------------------------------------------------------------------------------------
struct TapSharer {   // bounded search that lets lanes with the SAME start share a residue class (a broadcast)
  int lo[16], hi[16], choice[16], n;
  int cls_start[16];                 // start value owning residue class r, or -1
  std::vector<int> cls_lanes[16];

  bool place(int l, int depth, unsigned banned) {
    for (int s = hi[l]; s >= lo[l]; --s) {
      const int r = s & 15;
      if (banned & (1u << r)) continue;
      if (cls_start[r] < 0) { cls_start[r] = s; cls_lanes[r].assign(1, l); choice[l] = s; return true; }
      if (cls_start[r] == s) { cls_lanes[r].push_back(l); choice[l] = s; return true; }
    }
    if (depth >= 3) return false;
    for (int s = hi[l]; s >= lo[l]; --s) {
      const int r = s & 15;
      if (banned & (1u << r)) continue;
      const int old_start = cls_start[r];
      const std::vector<int> old_lanes = cls_lanes[r];
      cls_start[r] = s; cls_lanes[r].assign(1, l); choice[l] = s;
      bool ok = true;
      std::vector<int> seated;
      for (int x : old_lanes) {
        if (place(x, depth + 1, banned | (1u << r))) seated.push_back(x);
        else { ok = false; break; }
      }
      if (ok) return true;
      for (int x : seated) {             // undo
        const int rr = choice[x] & 15;
        std::vector<int>& v = cls_lanes[rr];
        for (size_t q = 0; q < v.size(); ++q) if (v[q] == x) { v.erase(v.begin() + q); break; }
        if (v.empty()) cls_start[rr] = -1;
      }
      cls_start[r] = old_start; cls_lanes[r] = old_lanes;
      for (int x : old_lanes) choice[x] = old_start;
    }
    return false;
  }
  bool run() {
    for (int r = 0; r < 16; ++r) { cls_start[r] = -1; cls_lanes[r].clear(); }
    for (int l = 0; l < n; ++l) if (!place(l, 0, 0u)) return false;
    return true;
  }
};

struct TapPlacer {   // bipartite matching lanes -> residue classes (Kuhn's augmenting paths; 16 x 16, so exact and tiny)
  int lo[16], hi[16], choice[16], n;
  int owner[16];                     // lane holding residue class r, or -1

  bool seat(int l, unsigned& visited) {
    const int span = hi[l] - lo[l] + 1;
    for (int d = 0; d < span && d < 16; ++d) {          // latest start first: fewest leading zero weights
      const int s = hi[l] - d, r = s & 15;
      if (visited & (1u << r)) continue;
      visited |= 1u << r;
      if (owner[r] < 0 || seat(owner[r], visited)) {
        owner[r] = l;
        choice[l] = s;
        return true;
      }
    }
    return false;
  }
  bool run() {
    for (int r = 0; r < 16; ++r) owner[r] = -1;
    for (int l = 0; l < n; ++l) {
      unsigned visited = 0u;
      if (!seat(l, visited)) return false;
    }
    return true;
  }
};

struct MelPlan {
  int first[kMaxMels], len[kMaxMels];   // slot m's run of FFT bins (segment m+1; slot 0 also takes segment 0)
  int start[kMaxMels];                  // first power bin the lane reads (<= first[m])
  int band_steps[kBands];
  int total_steps;
  std::vector<float> w;                 // [total_steps][16 lanes][2] = (wa, wb), bands back to back, unscaled
};

// starts and steps per band; falls back to start = first (correct, bank-conflicted) if the search fails
static void place_taps(int n_mels, MelPlan& mp) {
  for (int b = 0; b < kBands; ++b) {
    mp.band_steps[b] = 0;
    const int m0 = 16 * b, m1 = (n_mels < m0 + 16) ? n_mels : m0 + 16;
    if (m1 <= m0) continue;
    int mx = 1;
    for (int m = m0; m < m1; ++m) mx = mp.len[m] > mx ? mp.len[m] : mx;
    bool done = false;
    for (int T = mx; T <= mx + 8 && !done; ++T) {
      TapPlacer tp;
      tp.n = m1 - m0;
      for (int m = m0; m < m1; ++m) {
        int lo, hi;
        if (mp.len[m] == 0) {            // nothing to read: any start inside the power array will do
          lo = 0;
          hi = kBins - T;
        } else {
          lo = mp.first[m] + mp.len[m] - T;
          hi = mp.first[m];
          if (hi > kBins - T && kBins - T >= lo) hi = kBins - T;   // stay inside the 257 bins when the slack allows
        }
        tp.lo[m - m0] = lo > 0 ? lo : 0;
        tp.hi[m - m0] = hi > 0 ? hi : 0;
      }
      TapSharer ts;
      ts.n = tp.n;
      for (int l = 0; l < tp.n; ++l) { ts.lo[l] = tp.lo[l]; ts.hi[l] = tp.hi[l]; }
      const int* choice = nullptr;
      if (tp.run()) choice = tp.choice;
      else if (ts.run()) choice = ts.choice;
      if (choice) {
        for (int m = m0; m < m1; ++m) mp.start[m] = choice[m - m0];
        mp.band_steps[b] = T;
        done = true;
      }
    }
    if (!done) {
      for (int m = m0; m < m1; ++m) mp.start[m] = mp.first[m];
      mp.band_steps[b] = mx;
    }
  }
}

// dense (n_mels x 257) bank -> segment plan; LIDFE_E_MELBANK unless every bin feeds at most two ADJACENT filters and
// the plan reproduces the bank exactly
static int build_mel_plan(int n_mels, const float* bank, MelPlan& mp) {
  auto at = [&](int f, int k) { return bank[static_cast<size_t>(f) * kBins + k]; };
  std::vector<int> peak(n_mels, -1), seg(kBins, -1);
  for (int f = 0; f < n_mels; ++f) {
    float best = 0.f;
    for (int k = 0; k < kBins; ++k)
      if (at(f, k) > best) { best = at(f, k); peak[f] = k; }
    if (peak[f] < 0) return LIDFE_E_MELBANK;               // empty (or non-positive) row
  }
  for (int k = 0; k < kBins; ++k) {
    int lo = -1, n = 0, hi = -1;
    for (int f = 0; f < n_mels; ++f)
      if (at(f, k) != 0.f) { if (lo < 0) lo = f; hi = f; ++n; }
    if (n == 0) continue;
    if (n > 2 || hi - lo + 1 != n) return LIDFE_E_MELBANK;
    seg[k] = (n == 2) ? hi : (k <= peak[lo] ? lo : lo + 1);   // a lone weight: up-slope left of the peak, down-slope right
  }
  for (int m = 0; m < kMaxMels; ++m) mp.first[m] = mp.len[m] = mp.start[m] = 0;
  for (int m = 0; m < n_mels; ++m) {
    int first = -1, last = -1, cnt = 0;
    for (int k = 0; k < kBins; ++k)
      if (seg[k] == m + 1 || (m == 0 && seg[k] == 0)) { if (first < 0) first = k; last = k; ++cnt; }
    if (cnt == 0) continue;
    if (last - first + 1 != cnt || cnt > 64) return LIDFE_E_MELBANK;   // the run must be contiguous
    mp.first[m] = first;
    mp.len[m] = cnt;
  }
  place_taps(n_mels, mp);
  mp.total_steps = 0;
  for (int b = 0; b < kBands; ++b) mp.total_steps += mp.band_steps[b];
  mp.w.assign(static_cast<size_t>(mp.total_steps > 0 ? mp.total_steps : 1) * 32, 0.f);
  std::vector<float> recon(static_cast<size_t>(n_mels) * kBins, 0.f);
  int off = 0;
  for (int b = 0; b < kBands; ++b) {
    for (int t = 0; t < 16; ++t) {
      const int m = t + 16 * b;
      if (m >= n_mels) continue;
      for (int i = 0; i < mp.len[m]; ++i) {
        const int k = mp.first[m] + i;
        const float wa = at(m, k);
        const float wb = (m + 1 < n_mels && seg[k] == m + 1) ? at(m + 1, k) : 0.f;
        const size_t e = ((static_cast<size_t>(off) + (mp.first[m] - mp.start[m]) + i) * 16 + t) * 2;
        mp.w[e] = wa;
        mp.w[e + 1] = wb;
        recon[static_cast<size_t>(m) * kBins + k] += wa;
        if (m + 1 < n_mels) recon[static_cast<size_t>(m + 1) * kBins + k] += wb;
      }
    }
    off += mp.band_steps[b];
  }
  for (size_t i = 0; i < recon.size(); ++i)
    if (recon[i] != bank[i]) return LIDFE_E_MELBANK;
  return LIDFE_OK;
}

extern "C" {

int lidfe_abi_version(void) { return LIDFE_ABI_VERSION; }
long long lidfe_launch_count(void) { return g_launches.load(); }

// ---- host-side packer: B utterance buffers -> one packed (pinned) staging buffer -------------------------------------
// The reference's collate builds its batch with pad_sequence on the host (ref: lid/raw_datasets.py:345-351); here the
// host only gathers the raw samples at the plan's offsets.  A 256 x 1-20 s batch is 170 MB: one thread copies it at
// 5-8 GB/s, which would make the packer -- not PCIe, not the kernel -- the slowest stage of the ragged end-to-end path,
// so the byte range is cut into equal shares and copied by `threads` threads (utterances are split where a share ends).
int lidfe_pack_host(void* dst_host, const void* const* src_host, const long long* offsets, const long long* lengths,
                    int B, int elem_bytes, long long total_elems, int threads) {
  if (!dst_host || !src_host || !offsets || !lengths) return LIDFE_E_NULL;
  if (B <= 0 || (elem_bytes != 2 && elem_bytes != 4) || total_elems < 0) return LIDFE_E_ARG;
  long long pos = 0;
  for (int i = 0; i < B; ++i) {
    if (!src_host[i] && lengths[i] > 0) return LIDFE_E_NULL;
    if (lengths[i] < 0 || offsets[i] < pos || offsets[i] + lengths[i] > total_elems) return LIDFE_E_OFFSETS;
    pos = offsets[i] + lengths[i];
  }
  unsigned char* const dst = static_cast<unsigned char*>(dst_host);
  const long long eb = elem_bytes;
  // alignment gaps between utterances (and the tail) are zeroed so the staging buffer is a function of the batch alone
  auto work = [&](long long lo, long long hi) {          // bytes [lo, hi) of the packed buffer
    long long prev_end = 0;
    for (int i = 0; i < B; ++i) {
      const long long a = offsets[i] * eb, b = (offsets[i] + lengths[i]) * eb;
      const long long g0 = prev_end > lo ? prev_end : lo, g1 = a < hi ? a : hi;
      if (g1 > g0) memset(dst + g0, 0, static_cast<size_t>(g1 - g0));
      const long long c0 = a > lo ? a : lo, c1 = b < hi ? b : hi;
      if (c1 > c0) memcpy(dst + c0, static_cast<const unsigned char*>(src_host[i]) + (c0 - a), static_cast<size_t>(c1 - c0));
      prev_end = b;
      if (a >= hi) return;
    }
    const long long g0 = prev_end > lo ? prev_end : lo;
    if (hi > g0) memset(dst + g0, 0, static_cast<size_t>(hi - g0));
  };
  const long long total = total_elems * eb;
  int T = threads > 0 ? threads : static_cast<int>(std::thread::hardware_concurrency());
  if (T < 1) T = 1;
  if (T > 32) T = 32;
  if (total < (1ll << 20)) T = 1;
  if (T == 1) {
    work(0, total);
    return LIDFE_OK;
  }
  const long long share = ((total + T - 1) / T + 63) / 64 * 64;
  std::vector<std::thread> pool;
  try {
    for (int k = 1; k < T; ++k) {
      const long long lo = share * k, hi = (share * (k + 1) < total) ? share * (k + 1) : total;
      if (lo < hi) pool.emplace_back(work, lo, hi);
    }
  } catch (...) {
    for (auto& th : pool) th.join();
    work(0, total);                                      // could not start the threads: do all of it here
    return LIDFE_OK;
  }
  work(0, share < total ? share : total);
  for (auto& th : pool) th.join();
  return LIDFE_OK;
}

// Pinned sources need no staging copy at all: one cudaMemcpyAsync per utterance, straight to its place in the packed
// device buffer (a DataLoader with pin_memory=True hands out exactly such tensors).
// Zero-copy gather: the SMs read the pinned host buffers themselves (UVA: cudaHostAlloc'ed memory is mapped into the device's
// address space) and write the packed device buffer.  One launch per <= kGatherMax utterances replaces as many
// cudaMemcpyAsync calls, whose ~4.5 us of per-copy set-up on the copy engine held 256 copies of ~0.7 MB at 39 GB/s
// (4.5 ms per 174 MB batch); thousands of 16-byte loads in flight keep the link busy instead.
constexpr int kGatherMax = 120;
struct GatherArgs {
  const void* src[kGatherMax];
  long long off[kGatherMax];      // bytes into dst (16-byte aligned)
  long long len[kGatherMax];      // bytes
};
__global__ void __launch_bounds__(256) h2d_gather_kernel(unsigned char* __restrict__ dst, const __grid_constant__ GatherArgs A) {
  const int u = blockIdx.y;
  const unsigned char* src = static_cast<const unsigned char*>(A.src[u]);
  unsigned char* d = dst + A.off[u];
  const long long bytes = A.len[u];
  const long long n16 = bytes >> 4;
  const uint4* s4 = reinterpret_cast<const uint4*>(src);
  uint4* d4 = reinterpret_cast<uint4*>(d);
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n16; i += 4 * stride) {       // four independent 16-byte loads in flight per thread
    const uint4 a = s4[i], b = s4[i + stride], c = s4[i + 2 * stride], e = s4[i + 3 * stride];
    d4[i] = a; d4[i + stride] = b; d4[i + 2 * stride] = c; d4[i + 3 * stride] = e;
  }
  for (; i < n16; i += stride) d4[i] = s4[i];
  if (blockIdx.x == 0) {
    const long long tail0 = n16 << 4;
    for (long long j = tail0 + threadIdx.x; j < bytes; j += blockDim.x) d[j] = src[j];
  }
}

int lidfe_h2d_gather(void* dst_dev, const void* const* src_host, const long long* offsets, const long long* lengths,
                     int B, int elem_bytes, void* stream) {
  if (!dst_dev || !src_host || !offsets || !lengths) return LIDFE_E_NULL;
  if (B <= 0 || (elem_bytes != 2 && elem_bytes != 4)) return LIDFE_E_ARG;
  long long pos = 0;
  for (int i = 0; i < B; ++i) {
    if (!src_host[i] && lengths[i] > 0) return LIDFE_E_NULL;
    if (lengths[i] < 0 || offsets[i] < pos) return LIDFE_E_OFFSETS;
    pos = offsets[i] + lengths[i];
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned char* const dst = static_cast<unsigned char*>(dst_dev);
  // kernel path: every source 16-byte aligned and device-accessible, every destination 16-byte aligned
  bool kernel_ok = B >= 4 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  for (int i = 0; i < B && kernel_ok; ++i)
    kernel_ok = (reinterpret_cast<uintptr_t>(src_host[i]) & 15) == 0 && ((offsets[i] * elem_bytes) & 15) == 0;
  for (int k = 0; k < B && kernel_ok; ++k) {       // (~0.5 us per query: a source the device cannot read would be a fault, not an error code)
    cudaPointerAttributes at;
    const void* p = src_host[k];
    if (!p) continue;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); kernel_ok = false; break; }
    kernel_ok = (at.type == cudaMemoryTypeHost) && at.devicePointer == p;
  }
  if (kernel_ok) {
    for (int i0 = 0; i0 < B; i0 += kGatherMax) {
      GatherArgs A;
      const int n = B - i0 < kGatherMax ? B - i0 : kGatherMax;
      for (int i = 0; i < kGatherMax; ++i) {
        const bool live = i < n;
        A.src[i] = live ? src_host[i0 + i] : nullptr;
        A.off[i] = live ? offsets[i0 + i] * elem_bytes : 0;
        A.len[i] = live ? lengths[i0 + i] * elem_bytes : 0;
      }
      h2d_gather_kernel<<<dim3(16, static_cast<unsigned>(n)), 256, 0, st>>>(dst, A);
      g_launches.fetch_add(1);
      CU_TRY(cudaGetLastError());
    }
    return LIDFE_OK;
  }
  for (int i = 0; i < B; ++i) {
    if (lengths[i] == 0) continue;
    CU_TRY(cudaMemcpyAsync(dst + offsets[i] * elem_bytes, src_host[i], static_cast<size_t>(lengths[i]) * elem_bytes,
                           cudaMemcpyHostToDevice, st));
  }
  return LIDFE_OK;
}

int lidfe_stft_mel_db(const float* g_dev, const long long* g_off_dev, const long long* frames_dev, int B, long long max_frames,
                      int nw, const float* melT_dev, const int* mel_lo_dev, const int* mel_hi_dev, int n_bins, int n_mels,
                      float amin, float* out_dev, const long long* out_row_dev, double* stats_dev, int normalize, void* stream) {
  if (!g_dev || !g_off_dev || !frames_dev || !melT_dev || !mel_lo_dev || !mel_hi_dev || !out_dev || !out_row_dev || !stats_dev)
    return LIDFE_E_NULL;
  if (B <= 0 || B > 65535 || max_frames < 0 || nw < 2 * n_bins || (nw & 1) || n_bins < 2 || n_bins > kSfMaxBins || n_mels < 1)
    return LIDFE_E_ARG;
  if (max_frames == 0) return LIDFE_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CU_TRY(cudaMemsetAsync(stats_dev, 0, static_cast<size_t>(B) * 2 * sizeof(double), st));
  StftMelParams M;
  M.g = g_dev; M.g_off = g_off_dev; M.frames = frames_dev; M.out = out_dev; M.out_row = out_row_dev;
  M.melT = melT_dev; M.mel_lo = mel_lo_dev; M.mel_hi = mel_hi_dev; M.stats = stats_dev;
  M.nw = nw; M.n_bins = n_bins; M.n_mels = n_mels; M.amin = amin;
  const long long gx = (max_frames + kSfWarps - 1) / kSfWarps;
  if (gx > 0x7fffffffLL) return LIDFE_E_ARG;
  stft_mel_db_kernel<<<dim3(static_cast<unsigned>(gx), static_cast<unsigned>(B)), kSfWarps * 32, 0, st>>>(M);
  g_launches.fetch_add(1);
  CU_TRY(cudaGetLastError());
  if (normalize) {
    ScalarNormParams N;
    N.out = out_dev; N.out_row = out_row_dev; N.frames = frames_dev; N.stats = stats_dev; N.n_mels = n_mels;
    long long chunks = (max_frames * n_mels + 256 * 8 - 1) / (256 * 8);
    if (chunks < 1) chunks = 1;
    if (chunks > 4096) chunks = 4096;
    scalar_norm_kernel<<<dim3(static_cast<unsigned>(chunks), static_cast<unsigned>(B)), 256, 0, st>>>(N);
    g_launches.fetch_add(1);
    CU_TRY(cudaGetLastError());
  }
  return LIDFE_OK;
}

const char* lidfe_strerror(int rc) {
  switch (rc) {
    case LIDFE_OK: return "ok";
    case LIDFE_E_NULL: return "lidfe: required pointer is NULL";
    case LIDFE_E_CONFIG: return "lidfe: unsupported front-end configuration (need 16 kHz, 400/160/512 framing, 4<=n_mels<=80)";
    case LIDFE_E_SHORT: return "lidfe: utterance shorter than one frame (choose a window size that is [2, len])";
    case LIDFE_E_OFFSETS: return "lidfe: bad segment offsets";
    case LIDFE_E_ARG: return "lidfe: bad argument";
    case LIDFE_E_MELBANK: return "lidfe: mel bank row empty or wider than supported";
    case LIDFE_E_NOMEM: return "lidfe: host allocation failed";
    default: break;
  }
  if (rc > 0) return cudaGetErrorString(static_cast<cudaError_t>(rc));
  return "lidfe: unknown error";
}

long long lidfe_num_frames(long long n_samples, const lidfe_config* cfg) {
  if (!cfg || cfg->frame_len <= 0 || cfg->frame_shift <= 0) return 0;
  if (cfg->framing == LIDFE_FRAMING_CENTER) {
    const long long L = n_samples + 2LL * cfg->pad;
    if (n_samples < 0 || L <= cfg->fft_len / 2) return 0;      // torch.stft: reflect padding must be < input length
    return 1 + L / cfg->frame_shift;
  }
  if (n_samples < cfg->frame_len) return 0;
  return 1 + (n_samples - cfg->frame_len) / cfg->frame_shift;
}

int lidfe_out_dim(lidfe_handle h) { return h ? h->n_out : 0; }

int lidfe_mel_plan(int n_mels, const float* melbank_host, int* first_bin_out, int* num_taps_out, int* start_out,
                   int* band_taps_out) {
  if (!melbank_host || !first_bin_out || !num_taps_out || !start_out || !band_taps_out) return LIDFE_E_NULL;
  if (n_mels < 4 || n_mels > kMaxMels) return LIDFE_E_CONFIG;
  MelPlan mp;
  const int rc = build_mel_plan(n_mels, melbank_host, mp);
  if (rc != LIDFE_OK) return rc;
  for (int m = 0; m < n_mels; ++m) {
    first_bin_out[m] = mp.first[m];
    num_taps_out[m] = mp.len[m];
    start_out[m] = mp.start[m];
  }
  for (int b = 0; b < kBands; ++b) band_taps_out[b] = mp.band_steps[b];
  return LIDFE_OK;
}

int lidfe_mel_plan_expand(int n_mels, const float* melbank_host, float* dense_out) {
  if (!melbank_host || !dense_out) return LIDFE_E_NULL;
  if (n_mels < 4 || n_mels > kMaxMels) return LIDFE_E_CONFIG;
  MelPlan mp;
  const int rc = build_mel_plan(n_mels, melbank_host, mp);
  if (rc != LIDFE_OK) return rc;
  // replay the kernel's loop: slot m adds wa * P[start + i] to filter m and wb * P[start + i] to filter m + 1
  for (size_t i = 0; i < static_cast<size_t>(n_mels) * kBins; ++i) dense_out[i] = 0.f;
  int off = 0;
  for (int b = 0; b < kBands; ++b) {
    for (int t = 0; t < 16; ++t) {
      const int m = t + 16 * b;
      if (m >= n_mels) continue;
      for (int i = 0; i < mp.band_steps[b]; ++i) {
        const int k = mp.start[m] + i;
        const float wa = mp.w[((static_cast<size_t>(off) + i) * 16 + t) * 2], wb = mp.w[((static_cast<size_t>(off) + i) * 16 + t) * 2 + 1];
        if (k >= kBins) {
          if (wa != 0.f || wb != 0.f) return LIDFE_E_MELBANK;
          continue;
        }
        dense_out[static_cast<size_t>(m) * kBins + k] += wa;
        if (wb != 0.f) {
          if (m + 1 >= n_mels) return LIDFE_E_MELBANK;
          dense_out[static_cast<size_t>(m + 1) * kBins + k] += wb;
        }
      }
    }
    off += mp.band_steps[b];
  }
  return LIDFE_OK;
}

int lidfe_create(lidfe_handle* out, const lidfe_config* cfg, const float* window_host, const float* melbank_host,
                 const float* dct_host, const float* lifter_host) {
  if (!out || !cfg || !window_host || !melbank_host) return LIDFE_E_NULL;
  *out = nullptr;
  if (cfg->sample_rate != 16000 || cfg->frame_len != kFrameLen || cfg->frame_shift != kFrameShift ||
      cfg->fft_len != kFftLen || cfg->n_mels < 4 || cfg->n_mels > kMaxMels || cfg->n_ceps < 0 ||
      cfg->n_ceps > cfg->n_mels || (cfg->in_dtype != LIDFE_IN_F32 && cfg->in_dtype != LIDFE_IN_I16) ||
      !(cfg->preemph >= 0.f && cfg->preemph <= 1.f) ||
      (cfg->framing != LIDFE_FRAMING_KALDI && cfg->framing != LIDFE_FRAMING_CENTER) || cfg->pad < 0 ||
      cfg->pad > 4096 || (cfg->framing == LIDFE_FRAMING_KALDI && cfg->pad != 0) ||
      (cfg->log_kind != LIDFE_LOG_NATURAL && cfg->log_kind != LIDFE_LOG_DB10) ||
      !(cfg->log_floor >= 1.17549435e-38f) ||   // a normal float: the kernel's log takes no denormals
      !(cfg->dither >= 0.f) || (cfg->dither > 0.f && cfg->framing != LIDFE_FRAMING_KALDI) ||
      cfg->window_type < LIDFE_WINDOW_POVEY || cfg->window_type > LIDFE_WINDOW_HANN_PERIODIC)
    return LIDFE_E_CONFIG;
  if (cfg->n_ceps > 0 && !dct_host) return LIDFE_E_NULL;

  lidfe_ctx* c = new (std::nothrow) lidfe_ctx();
  if (!c) return LIDFE_E_NOMEM;
  c->cfg = *cfg;
  c->n_out = cfg->n_ceps > 0 ? cfg->n_ceps : cfg->n_mels;

  // ---- dense bank -> segment plan (see build_mel_plan).  The kernel leaves the power bins scaled by 4 (it skips the
  //      1/2 of the real-FFT split), so the weights carry the exact factor 1/4.
  MelPlan mp;
  {
    const int rc = build_mel_plan(cfg->n_mels, melbank_host, mp);
    if (rc != LIDFE_OK) {
      delete c;
      return rc;
    }
  }
  const int total_taps = mp.total_steps;
  for (int b = 0; b < kBands; ++b) c->band_taps[b] = mp.band_steps[b];
  c->std_mel = 0;
  for (int kind = 1; kind <= 2 && !c->std_mel; ++kind) {
    bool same = true;
    for (int b = 0; b < kBands; ++b) same = same && (c->band_taps[b] == std_taps(kind, b));
    if (same && cfg->n_mels == 80) c->std_mel = kind;      // (the kernel variants hard-wire 80 output dims)
  }
  // the unrolled variants also hard-wire the framing of the call they belong to (see the kernel)
  if (c->std_mel == 1 && !(cfg->remove_dc && cfg->preemph == 1.f)) c->std_mel = 0;
  // ... and variant 1 the reference call's log: natural, floored at FLT_EPSILON (compile-time constants in the warp kernel)
  if (c->std_mel == 1 && !(cfg->log_kind == LIDFE_LOG_NATURAL && cfg->log_floor == 1.1920928955078125e-07f)) c->std_mel = 0;
  if (c->std_mel == 2 && !(!cfg->remove_dc && cfg->preemph == 0.f)) c->std_mel = 0;
  std::vector<float> melw(mp.w);
  for (float& v : melw) v *= 0.25f;
  std::vector<int> k0(mp.start, mp.start + kMaxMels);   // the kernel's per-lane first power bin

  // ---- twiddles, rounded once from fp64
  std::vector<float2> tw1(256), tw2(128);
  const double kPi = 3.14159265358979323846;
  for (int K1 = 0; K1 < 16; ++K1)
    for (int t = 0; t < 16; ++t) {
      const double a = -2.0 * kPi * static_cast<double>(K1 * t) / 256.0;
      tw1[K1 * 16 + t] = make_float2(static_cast<float>(cos(a)), static_cast<float>(sin(a)));
    }
  for (int i = 0; i < 8; ++i)
    for (int t = 0; t < 16; ++t) {
      const double a = -2.0 * kPi * static_cast<double>(t + 16 * i) / 512.0;
      tw2[i * 16 + t] = make_float2(static_cast<float>(cos(a)), static_cast<float>(sin(a)));
    }
  std::vector<float> window(416, 0.f);
  for (int i = 0; i < kFrameLen; ++i) window[i] = window_host[i];
  std::vector<float> lifter(cfg->n_ceps > 0 ? cfg->n_ceps : 1, 1.f);
  if (cfg->n_ceps > 0 && lifter_host)
    for (int i = 0; i < cfg->n_ceps; ++i) lifter[i] = lifter_host[i];

  // ---- one blob in the kernel's shared-memory table layout (every section a multiple of 16 bytes)
  std::vector<unsigned char> blob;
  auto append = [&blob](const void* src, size_t bytes) {
    const size_t at = blob.size();
    blob.resize(at + ((bytes + 15) & ~static_cast<size_t>(15)), 0);
    memcpy(blob.data() + at, src, bytes);
  };
  append(window.data(), window.size() * sizeof(float));
  append(tw1.data(), tw1.size() * sizeof(float2));
  append(tw2.data(), tw2.size() * sizeof(float2));
  c->k0_off = static_cast<int>(blob.size());
  append(k0.data(), static_cast<size_t>(kMaxMels) * sizeof(int));
  c->melw_off = static_cast<int>(blob.size());
  c->total_taps = total_taps;
  if (total_taps > 0) append(melw.data(), static_cast<size_t>(total_taps) * 32 * sizeof(float));
  c->blob_bytes_fbank = static_cast<int>(blob.size());
  if (cfg->n_ceps > 0) {
    c->dct_off = static_cast<int>(blob.size());
    append(dct_host, static_cast<size_t>(cfg->n_mels) * cfg->n_ceps * sizeof(float));
    c->lifter_off = static_cast<int>(blob.size());
    append(lifter.data(), static_cast<size_t>(cfg->n_ceps) * sizeof(float));
  }
  c->blob_bytes = static_cast<int>(blob.size());

  // test selector: LIDFE_WARP_KERNEL=0 keeps fbank_kernel, the reference the warp kernel is tested against
  if (const char* env = getenv("LIDFE_WARP_KERNEL")) c->warp_off = atoi(env) == 0;
  cudaError_t e = cudaGetDevice(&c->device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, c->device);
  if (e == cudaSuccess) e = upload(&c->d_blob, blob.data(), blob.size());
  if (e == cudaSuccess) e = cudaDeviceSynchronize();   // the tables have landed whatever stream the caller launches on
  if (e == cudaSuccess) {
    c->smem_bytes = smem_for(*cfg, total_taps);
    if (handle_has_dct_path(c)) {
      // two-kernel MFCC path: fbank-only variant into a log-mel workspace, then mfcc_dct_mma_kernel
      lidfe_config fb = *cfg;
      fb.n_ceps = 0;
      c->smem_bytes_fbank = smem_for(fb, total_taps);
      e = cudaFuncSetAttribute(pick_kernel(cfg->in_dtype, false, c->std_mel), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               static_cast<int>(c->smem_bytes_fbank));
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(mfcc_dct_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMmSmemBytes);
    }
    fbank_fn fn = pick_kernel(cfg->in_dtype, cfg->n_ceps > 0, c->std_mel);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(c->smem_bytes));
    if (e == cudaSuccess) {
      int per_sm = 0;
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kThreads, c->smem_bytes);
      if (e == cudaSuccess) {
        if (per_sm < 1) per_sm = 1;
        c->grid_cap = per_sm * c->num_sms;
      }
    }
  }
  if (e == cudaSuccess && handle_can_warp(c)) {
    c->w_tab_bytes = static_cast<int>((kWTabOff + c->blob_bytes_fbank + kMaxMels * 8 + 127) / 128 * 128);
    const size_t per_warp = (cfg->in_dtype == LIDFE_IN_I16) ? WarpLayout<short>::kWarpBytes : WarpLayout<float>::kWarpBytes;
    c->w_smem = static_cast<size_t>(c->w_tab_bytes) + kWWarps * per_warp;
    fbank_fn wf = pick_warp_kernel(cfg->in_dtype, c->std_mel, 1);
    e = cudaFuncSetAttribute(wf, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(c->w_smem));
    for (int sk = 0; sk <= 2 && e == cudaSuccess; sk += 2)
      e = cudaFuncSetAttribute(pick_warp_kernel(cfg->in_dtype, c->std_mel, sk), cudaFuncAttributeMaxDynamicSharedMemorySize,
                               static_cast<int>(c->w_smem));
    if (e == cudaSuccess) {
      int per_sm = 0;
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wf, kWThreads, c->w_smem);
      if (e == cudaSuccess) c->w_grid = (per_sm < 1 ? 1 : per_sm) * c->num_sms;
    }
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    lidfe_destroy(c);
    return static_cast<int>(e);
  }
  *out = c;
  return LIDFE_OK;
}

static void free_block(PlanBlock* b) {
  if (!b) return;
  cudaFree(b->d_base);
  cudaFreeHost(b->h_tables);
  cudaFree(b->d_logmel);
  if (b->ev) cudaEventDestroy(b->ev);
  delete b;
}

static void destroy_now(lidfe_ctx* h) {
  cudaFree(h->d_blob);
  for (PlanBlock* b : h->pool) free_block(b);
  for (cudaEvent_t ev : h->prof_events) cudaEventDestroy(ev);
  delete h;
}

// A handle may be destroyed before its plans (garbage-collected bindings give no order): the plans keep it alive
// and the last one to go frees it.
int lidfe_destroy(lidfe_handle h) {
  if (!h) return LIDFE_E_NULL;
  {
    std::lock_guard<std::mutex> g(h->pool_mu);
    if (h->live_plans > 0) {
      h->destroyed = true;
      return LIDFE_OK;
    }
  }
  destroy_now(h);
  return LIDFE_OK;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
struct BlockLayout {
  size_t sched, utt_max, utt_min, utt_stats, utt_wnorm, ws_bytes;
  size_t frames, out_rows, offsets, lengths, first_tile, spans, wfirst, wspans, tiles, tab_bytes;   // tables: relative to ws_bytes
};
static BlockLayout block_layout(int Bc, long long Sc, long long Tc, long long Wc, int n_out, long long n_warps) {
  BlockLayout L;
  size_t o = 0;
  L.sched = o; o += 16;
  L.utt_max = o; o = align_up(o + 2 * static_cast<size_t>(Bc) * 4, 16);          // [2 launch parities][Bc]
  L.utt_min = o; o = align_up(o + 2 * static_cast<size_t>(Bc) * 4, 16);
  L.utt_stats = o; o = align_up(o + 2 * static_cast<size_t>(Bc) * 2 * n_out * 8, 16);
  L.utt_wnorm = o; o = align_up(o + static_cast<size_t>(Bc) * 8, 256);
  L.ws_bytes = o;
  o = 0;
  L.frames = o; o += static_cast<size_t>(Bc) * 8;
  L.out_rows = o; o += static_cast<size_t>(Bc) * 8;
  L.offsets = o; o += static_cast<size_t>(Bc) * 8;
  L.lengths = o; o += static_cast<size_t>(Bc) * 8;
  L.first_tile = o; o = align_up(o + static_cast<size_t>(Bc) * 8, 32);
  L.spans = o; o += static_cast<size_t>(Sc) * sizeof(Span);
  L.wfirst = o; o = align_up(o + (Wc > 0 ? static_cast<size_t>(n_warps) + 1 : 0) * 4, 32);
  L.wspans = o; o += static_cast<size_t>(Wc) * sizeof(Span);
  L.tiles = o; o += static_cast<size_t>(Tc) * sizeof(Tile);
  L.tab_bytes = align_up(o, 256);
  return L;
}
static long long pow2_at_least(long long v, long long lo) {
  long long c = lo;
  while (c < v) c <<= 1;
  return c;
}

// a block with room for (B, spans, tiles): from the pool if one fits, else a new allocation (the only place that
// allocates; the workspace is put to rest once, here -- the kernels leave it at rest)
static int acquire_block(lidfe_ctx* h, int B, long long n_spans, long long n_tiles, long long n_wspans, PlanBlock** out) {
  *out = nullptr;
  {
    // first choice: a block that fits and whose previous work has finished (no waiting); second: while the handle owns
    // fewer than kPoolAsyncBlocks blocks, a new one (so that a loop that creates and destroys a plan per batch can run
    // ahead of the device); last: wait for a busy block that fits
    constexpr long long kPoolAsyncBlocks = 4;
    std::lock_guard<std::mutex> g(h->pool_mu);
    int busy = -1;
    for (size_t i = 0; i < h->pool.size(); ++i) {
      PlanBlock* b = h->pool[i];
      if (b->Bc >= B && b->Sc >= n_spans && b->Tc >= n_tiles && b->Wc >= n_wspans) {
        if (cudaEventQuery(b->ev) == cudaSuccess) {
          h->pool.erase(h->pool.begin() + i);
          *out = b;
          break;
        }
        cudaGetLastError();
        if (busy < 0) busy = static_cast<int>(i);
      }
    }
    if (!*out && busy >= 0 && h->blocks_allocated >= kPoolAsyncBlocks) {
      *out = h->pool[busy];
      h->pool.erase(h->pool.begin() + busy);
    }
  }
  if (*out) {
    CU_TRY(cudaEventSynchronize((*out)->ev));     // its previous plan's work (normally long done)
    return LIDFE_OK;
  }
  PlanBlock* b = new (std::nothrow) PlanBlock();
  if (!b) return LIDFE_E_NOMEM;
  memset(b, 0, sizeof(*b));
  b->Bc = static_cast<int>(pow2_at_least(B, 64));
  b->Sc = pow2_at_least(n_spans, 256);
  b->Tc = n_tiles > 0 ? pow2_at_least(n_tiles, 256) : 0;
  b->Wc = n_wspans > 0 ? pow2_at_least(n_wspans, 256) : 0;
  const BlockLayout L = block_layout(b->Bc, b->Sc, b->Tc, b->Wc, h->n_out, static_cast<long long>(h->w_grid) * kWWarps);
  b->ws_bytes = L.ws_bytes;
  b->tab_bytes = L.tab_bytes;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&b->d_base), L.ws_bytes + L.tab_bytes);
  if (e == cudaSuccess) e = cudaMallocHost(reinterpret_cast<void**>(&b->h_tables), L.tab_bytes);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaMemset(b->d_base, 0, L.ws_bytes);
  if (e == cudaSuccess) e = cudaMemset(b->d_base + L.utt_min, 0xff, 2 * static_cast<size_t>(b->Bc) * 4);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cudaGetLastError();
    free_block(b);
    return static_cast<int>(e);
  }
  {
    std::lock_guard<std::mutex> g(h->pool_mu);
    ++h->blocks_allocated;
  }
  *out = b;
  return LIDFE_OK;
}

constexpr int kZeroRows = 4 * kTileFrames;   // output rows one zero-fill span clears

// The spans of a plan, for both kernels' lists: where a run of frames of utterance i starts in the packed input, and
// whether its samples may be bulk-copied (aux = 1): the first sample inside the buffer on a 16-byte boundary and, for
// the warp kernel's quads under CENTER framing, none of them in the padding / reflection (`interior`).
struct SpanMaker {
  const long long* offsets;
  const long long* out_rows;
  long long in_elt, pad;
  bool center;
  // first sample of frame f relative to the utterance's first.  CENTER framing: frame f covers p[160 f - 200, 160 f + 200)
  // of the constant-padded signal p (the Hann window sits at 56..455 of the 512-point buffer and |FFT|^2 does not see
  // that shift)
  long long rel(long long f) const { return center ? f * kFrameShift - kFrameLen / 2 - pad : f * kFrameShift; }
  // the quad starting at frame q0 (<= 4 frames, never past the utterance's T-th) reads only the utterance's N samples
  bool quad_interior(long long q0, long long T, long long N) const {
    const long long fr = (T - q0) < kQuadFrames ? (T - q0) : kQuadFrames;
    return rel(q0) >= 0 && rel(q0) + fr * kFrameShift + (kFrameLen - kFrameShift) <= N;
  }
  Span frames(int i, long long f, long long nf, bool interior) const {
    Span sp;
    sp.wav_off = offsets[i] + rel(f);
    sp.out_row = out_rows[i] + f;
    sp.nframes = static_cast<int>(nf);
    sp.utt = i;
    sp.t0 = static_cast<int>(f);
    sp.aux = (interior && sp.wav_off >= 0 && (sp.wav_off * in_elt) % 16 == 0) ? 1 : 0;
    return sp;
  }
  // pad_sequence's zeros behind utterance i's T frames (ref: lid/raw_datasets.py:347-350): spans of no frames that
  // clear up to kZeroRows rows each (aux = rows)
  void zero_fill(std::vector<Span>& dst, int i, long long T, long long pad_rows) const {
    for (long long r = T; r < pad_rows; r += kZeroRows) {
      Span sp;
      sp.wav_off = 0;
      sp.out_row = out_rows[i] + r;
      sp.nframes = 0;
      sp.utt = i;
      sp.t0 = static_cast<int>(r);
      sp.aux = static_cast<int>(pad_rows - r < kZeroRows ? pad_rows - r : kZeroRows);
      dst.push_back(sp);
    }
  }
};

int lidfe_plan_create_async(lidfe_handle h, lidfe_plan* out, int B, const long long* wav_offsets_host,
                            const long long* wav_lengths_host, const long long* out_rows_host,
                            const long long* pad_rows_host, void* stream) {
  if (!h || !out || !wav_offsets_host || !wav_lengths_host || !out_rows_host) return LIDFE_E_NULL;
  *out = nullptr;
  if (B <= 0) return LIDFE_E_ARG;
  const SpanMaker mk = {wav_offsets_host, out_rows_host, (h->cfg.in_dtype == LIDFE_IN_I16) ? 2 : 4, h->cfg.pad,
                       h->cfg.framing == LIDFE_FRAMING_CENTER};
  const bool dct_path = handle_has_dct_path(h);
  std::vector<long long> frames(B), utt_first_tile(B);
  long long total = 0, n_tiles = 0, max_frames = 0;
  for (int i = 0; i < B; ++i) {
    if (wav_offsets_host[i] < 0 || out_rows_host[i] < 0) return LIDFE_E_OFFSETS;
    const long long T = lidfe_num_frames(wav_lengths_host[i], &h->cfg);
    if (T <= 0) return LIDFE_E_SHORT;
    if (T > 0x7fffffffLL) return LIDFE_E_ARG;
    if (pad_rows_host && pad_rows_host[i] < T) return LIDFE_E_OFFSETS;
    frames[i] = T;
    total += T;
    max_frames = T > max_frames ? T : max_frames;
    utt_first_tile[i] = n_tiles;
    n_tiles += (T + kTileFrames - 1) / kTileFrames;
    if (pad_rows_host && dct_path) n_tiles += (pad_rows_host[i] - T + kZeroRows - 1) / kZeroRows;
  }
  if (n_tiles > 0x7fffffffLL) return LIDFE_E_ARG;

  // ---- spans: runs of <= span_tiles consecutive tiles of one utterance, utterance-major.  Enough spans per CTA that
  //      dynamic claiming balances (>= ~10), as long as possible otherwise (a span end costs two CTA barriers, and in
  //      the per-utterance modes a hand-over of 2 x n_out sums); the spans of the last stretch of the batch are single
  //      tiles so that the CTAs run dry together.  Under CENTER framing fbank_kernel decides per tile which ones touch
  //      the padding / reflection and stages those element-wise.
  const long long per_cta_tiles = n_tiles / (h->grid_cap > 0 ? h->grid_cap : 1);
  int span_tiles = static_cast<int>(per_cta_tiles / 10);
  if (span_tiles < 1) span_tiles = 1;
  if (span_tiles > kMaxSpanTiles) span_tiles = kMaxSpanTiles;
  const long long tail_tiles = static_cast<long long>(h->grid_cap) * span_tiles;   // ~ one round of spans
  std::vector<Span> spans;
  std::vector<Tile> tiles;
  {
    long long tile_no = 0;
    for (int i = 0; i < B; ++i) {
      const long long T = frames[i];
      for (long long f = 0; f < T;) {
        const int st = (n_tiles - tile_no <= tail_tiles) ? 1 : span_tiles;
        const long long nf = (T - f) < static_cast<long long>(st) * kTileFrames ? (T - f) : static_cast<long long>(st) * kTileFrames;
        const Span sp = mk.frames(i, f, nf, true);
        spans.push_back(sp);
        if (dct_path) {
          for (long long g = f; g < f + nf; g += kTileFrames) {
            Tile tl = sp;
            tl.wav_off = sp.wav_off + (g - f) * kFrameShift;
            tl.out_row = out_rows_host[i] + g;
            tl.nframes = static_cast<int>((T - g) < kTileFrames ? (T - g) : kTileFrames);
            tl.t0 = static_cast<int>(g);
            tiles.push_back(tl);
          }
        }
        tile_no += (nf + kTileFrames - 1) / kTileFrames;
        f += nf;
      }
      if (pad_rows_host) {
        const size_t z = spans.size();
        mk.zero_fill(spans, i, T, pad_rows_host[i]);
        if (dct_path) tiles.insert(tiles.end(), spans.begin() + z, spans.end());
      }
    }
  }
  if (spans.size() > 0x7fffffffull) return LIDFE_E_ARG;

  lidfe_plan_s* p = new (std::nothrow) lidfe_plan_s();
  if (!p) return LIDFE_E_NOMEM;
  p->ctx = h;
  p->B = B;
  p->total_frames = total;
  p->n_tiles = n_tiles;
  p->n_spans = static_cast<long long>(spans.size());
  p->frames = frames;
  p->max_frames = max_frames;
  p->max_row = 0;
  for (int i = 0; i < B; ++i) {
    const long long end = out_rows_host[i] + ((pad_rows_host && pad_rows_host[i] > frames[i]) ? pad_rows_host[i] : frames[i]);
    if (end > p->max_row) p->max_row = end;
  }
  // ---- warp spans (lidfe_fbank_warp.cuh).  The quads (4 frames) of the batch, utterance-major, are dealt out as
  //      W contiguous STATIC runs of s = floor(0.9 Q / W) quads, one per warp (cut into spans where the utterance changes),
  //      followed by a POOL of one-quad spans (zero-fill runs first, then the last Q - W s quads) that the warps claim one at
  //      a time when their own run is done.  w_first[w] .. w_first[w + 1] are warp w's static spans.
  std::vector<Span> wspans;
  std::vector<int> w_first;
  bool all_aligned = true;
  for (int i = 0; i < B; ++i) all_aligned = all_aligned && ((wav_offsets_host[i] * mk.in_elt) % 16) == 0;
  if (plan_can_warp(h, all_aligned)) {
    long long n_quads = 0;
    for (int i = 0; i < B; ++i) n_quads += (frames[i] + kQuadFrames - 1) / kQuadFrames;
    const long long W = static_cast<long long>(h->w_grid) * kWWarps;
    const long long s_run = (n_quads * 90) / (100 * W);                     // static quads per warp
    const long long static_quads = s_run * W;
    std::vector<Span> pool;
    // CENTER framing: a run is cut so that the quads that touch the padding / the reflection -- the first quad of an
    // utterance and its last one or two -- are spans of their own with aux = 0 (staged element by element), everything
    // else stays on TMA
    auto push_frames = [&](std::vector<Span>& dst, int i, long long f, long long nf) {
      if (!mk.center) {
        dst.push_back(mk.frames(i, f, nf, true));
        return;
      }
      auto interior = [&](long long q0) { return mk.quad_interior(q0, frames[i], wav_lengths_host[i]); };
      long long g = f;
      while (g < f + nf) {                          // maximal runs of quads of one kind
        const bool in0 = interior(g);
        long long e = g + kQuadFrames;
        while (e < f + nf && interior(e) == in0) e += kQuadFrames;
        if (e > f + nf) e = f + nf;
        dst.push_back(mk.frames(i, g, e - g, in0));
        g = e;
      }
    };
    if (pad_rows_host)
      for (int i = 0; i < B; ++i) mk.zero_fill(pool, i, frames[i], pad_rows_host[i]);
    std::vector<std::vector<Span>> per_warp(static_cast<size_t>(W));
    long long quad_no = 0;      // quads dealt out so far
    for (int i = 0; i < B; ++i) {
      const long long T = frames[i];
      for (long long f = 0; f < T;) {
        const long long left_q = (T - f + kQuadFrames - 1) / kQuadFrames;        // quads left in this utterance
        if (quad_no < static_quads) {
          const long long k = quad_no / s_run;                                  // run being filled
          long long q = (k + 1) * s_run - quad_no;                              // quads left in this run
          if (q > left_q) q = left_q;
          const long long nf = (T - f) < q * kQuadFrames ? (T - f) : q * kQuadFrames;
          push_frames(per_warp[static_cast<size_t>(k)], i, f, nf);
          quad_no += q;
          f += nf;
        } else {
          const long long nf = (T - f) < kQuadFrames ? (T - f) : kQuadFrames;
          push_frames(pool, i, f, nf);
          quad_no += 1;
          f += nf;
        }
      }
    }
    w_first.assign(static_cast<size_t>(W) + 1, 0);
    for (long long w = 0; w < W; ++w) {
      w_first[static_cast<size_t>(w)] = static_cast<int>(wspans.size());
      wspans.insert(wspans.end(), per_warp[static_cast<size_t>(w)].begin(), per_warp[static_cast<size_t>(w)].end());
    }
    w_first[static_cast<size_t>(W)] = static_cast<int>(wspans.size());
    p->n_wstatic = static_cast<int>(wspans.size());
    wspans.insert(wspans.end(), pool.begin(), pool.end());
    if (wspans.size() > 0x7fffffffull) {
      delete p;
      return LIDFE_E_ARG;
    }
  }
  p->n_wspans = static_cast<long long>(wspans.size());
  p->all_aligned = all_aligned;
  PlanBlock* b = nullptr;
  const int rc = acquire_block(h, B, p->n_spans, static_cast<long long>(tiles.size()), p->n_wspans, &b);
  if (rc != LIDFE_OK) {
    delete p;
    return rc;
  }
  p->blk = b;
  {
    std::lock_guard<std::mutex> g(h->pool_mu);
    ++h->live_plans;
  }
  const BlockLayout L = block_layout(b->Bc, b->Sc, b->Tc, b->Wc, h->n_out, static_cast<long long>(h->w_grid) * kWWarps);
  unsigned char* ws = b->d_base;
  unsigned char* tab = b->d_base + L.ws_bytes;
  p->d_sched = reinterpret_cast<int*>(ws + L.sched);
  p->d_utt_max = reinterpret_cast<unsigned*>(ws + L.utt_max);
  p->d_utt_min = reinterpret_cast<unsigned*>(ws + L.utt_min);
  p->d_utt_stats = reinterpret_cast<double*>(ws + L.utt_stats);
  p->d_utt_wnorm = reinterpret_cast<float2*>(ws + L.utt_wnorm);
  p->d_frames = reinterpret_cast<long long*>(tab + L.frames);
  p->d_out_rows = reinterpret_cast<long long*>(tab + L.out_rows);
  p->d_offsets = reinterpret_cast<long long*>(tab + L.offsets);
  p->d_lengths = reinterpret_cast<long long*>(tab + L.lengths);
  p->d_utt_first_tile = reinterpret_cast<long long*>(tab + L.first_tile);
  p->d_spans = reinterpret_cast<Span*>(tab + L.spans);
  p->d_wspans = wspans.empty() ? nullptr : reinterpret_cast<Span*>(tab + L.wspans);
  p->d_w_first = wspans.empty() ? nullptr : reinterpret_cast<int*>(tab + L.wfirst);
  p->d_tiles = tiles.empty() ? nullptr : reinterpret_cast<Tile*>(tab + L.tiles);
  // fill the pinned mirror, ONE asynchronous copy of what is used
  unsigned char* ht = b->h_tables;
  memcpy(ht + L.frames, frames.data(), static_cast<size_t>(B) * 8);
  memcpy(ht + L.out_rows, out_rows_host, static_cast<size_t>(B) * 8);
  memcpy(ht + L.offsets, wav_offsets_host, static_cast<size_t>(B) * 8);
  memcpy(ht + L.lengths, wav_lengths_host, static_cast<size_t>(B) * 8);
  memcpy(ht + L.first_tile, utt_first_tile.data(), static_cast<size_t>(B) * 8);
  memcpy(ht + L.spans, spans.data(), spans.size() * sizeof(Span));
  if (!wspans.empty()) {
    memcpy(ht + L.wspans, wspans.data(), wspans.size() * sizeof(Span));
    memcpy(ht + L.wfirst, w_first.data(), w_first.size() * sizeof(int));
  }
  if (!tiles.empty()) memcpy(ht + L.tiles, tiles.data(), tiles.size() * sizeof(Tile));
  const size_t used = !tiles.empty() ? L.tiles + tiles.size() * sizeof(Tile)
                      : !wspans.empty() ? L.wspans + wspans.size() * sizeof(Span) : L.spans + spans.size() * sizeof(Span);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemcpyAsync(tab, ht, used, cudaMemcpyHostToDevice, st);
  // the workspace goes to rest (asynchronously, on the same stream): whatever the block's previous plan -- another
  // batch size, an aborted launch -- left behind cannot leak into this one
  if (e == cudaSuccess) e = cudaMemsetAsync(ws, 0, L.ws_bytes, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(ws + L.utt_min, 0xff, 2 * static_cast<size_t>(b->Bc) * 4, st);
  p->parity = 0;
  if (e == cudaSuccess) e = cudaEventRecord(b->ev, st);
  if (e != cudaSuccess) {
    cudaGetLastError();
    lidfe_plan_destroy(p);
    return static_cast<int>(e);
  }
  *out = p;
  return LIDFE_OK;
}

int lidfe_plan_create(lidfe_handle h, lidfe_plan* out, int B, const long long* wav_offsets_host,
                      const long long* wav_lengths_host, const long long* out_rows_host,
                      const long long* pad_rows_host) {
  const int rc = lidfe_plan_create_async(h, out, B, wav_offsets_host, wav_lengths_host, out_rows_host, pad_rows_host, nullptr);
  if (rc != LIDFE_OK) return rc;
  CU_TRY(cudaEventSynchronize((*out)->blk->ev));      // the tables have landed: the plan may be used on any stream
  return LIDFE_OK;
}

int lidfe_plan_destroy(lidfe_plan p) {
  if (!p) return LIDFE_E_NULL;
  lidfe_ctx* h = p->ctx;
  bool last = false;
  if (p->blk) {
    std::lock_guard<std::mutex> g(h->pool_mu);
    h->pool.push_back(p->blk);
    --h->live_plans;
    last = h->destroyed && h->live_plans == 0;
  }
  delete p;
  if (last) destroy_now(h);
  return LIDFE_OK;
}
int lidfe_pool_stats(lidfe_handle h, long long* blocks_allocated, long long* blocks_free) {
  if (!h || !blocks_allocated || !blocks_free) return LIDFE_E_NULL;
  std::lock_guard<std::mutex> g(h->pool_mu);
  *blocks_allocated = h->blocks_allocated;
  *blocks_free = static_cast<long long>(h->pool.size());
  return LIDFE_OK;
}
long long lidfe_plan_total_frames(lidfe_plan p) { return p ? p->total_frames : 0; }
long long lidfe_plan_num_tiles(lidfe_plan p) { return p ? p->n_tiles : 0; }
long long lidfe_plan_num_spans(lidfe_plan p) { return p ? p->n_spans : 0; }
long long lidfe_plan_frames(lidfe_plan p, int i) { return (p && i >= 0 && i < p->B) ? p->frames[i] : 0; }

static int launch_apply(lidfe_ctx* h, lidfe_plan p, float* feats, long long ld, const int* masks, int n_masks,
                        const double* glob_stats, cudaStream_t st, int normalize, int parity = -1) {
  ApplyParams A;
  memset(&A, 0, sizeof(A));
  A.feats = feats;
  A.ld = ld;
  A.n_out = h->n_out;
  A.masks = masks;
  A.n_masks = masks ? n_masks : 0;
  A.utt_stats = nullptr;
  A.utt_frames = p->d_frames;
  A.utt_out_row = p->d_out_rows;
  A.glob_stats = glob_stats;
  A.normalize = normalize;
  A.utt_max = p->d_utt_max;
  A.top_db = h->cfg.top_db;
  if (parity >= 0) {     // second kernel of a per-utterance mode: this launch's half in, the other half back to rest
    const long long Bc = p->blk->Bc;
    const int op = parity ^ 1;
    if (normalize == 1) A.utt_stats = p->d_utt_stats + static_cast<long long>(parity) * Bc * 2 * h->n_out;
    A.utt_max = p->d_utt_max + parity * Bc;
    A.utt_min = p->d_utt_min + parity * Bc;
    A.rest_stats = p->d_utt_stats + static_cast<long long>(op) * Bc * 2 * h->n_out;
    A.rest_max = p->d_utt_max + op * Bc;
    A.rest_min = p->d_utt_min + op * Bc;
  }
  A.rows_per_cta = kApplyRows;
  const long long chunks = (p->max_frames + A.rows_per_cta - 1) / A.rows_per_cta;
  if (chunks > 65535) return LIDFE_E_ARG;
  dim3 grid(static_cast<unsigned>(p->B), static_cast<unsigned>(chunks));
  cmvn_apply_kernel<<<grid, 256, 0, st>>>(A);
  g_launches.fetch_add(1);
  CU_TRY(cudaGetLastError());
  CU_TRY(cudaEventRecord(p->blk->ev, st));
  return LIDFE_OK;
}

// the wave_stages_kernel parameters every caller sets; the stages it does not name start off
static WaveParams wave_params(lidfe_plan p, const void* in, int in_i16, float in_scale, float* out, int normalize) {
  WaveParams W;
  memset(&W, 0, sizeof(W));
  W.in = in;
  W.in_i16 = in_i16;
  W.in_scale = in_scale;
  W.out = out;
  W.offsets = p->d_offsets;
  W.lengths = p->d_lengths;
  W.normalize = normalize;
  return W;
}

// noise: kNoiseNone / kNoiseBank / kNoiseGauss (the wave_stages_kernel instantiation)
static int run_wave(lidfe_plan p, const WaveParams& W, int noise, void* stream) {
  const dim3 grid(static_cast<unsigned>(p->B) * kWaveCluster);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (noise == kNoiseBank) wave_stages_kernel<kNoiseBank><<<grid, kWaveThreads, 0, st>>>(W);
  else if (noise == kNoiseGauss) wave_stages_kernel<kNoiseGauss><<<grid, kWaveThreads, 0, st>>>(W);
  else wave_stages_kernel<kNoiseNone><<<grid, kWaveThreads, 0, st>>>(W);
  g_launches.fetch_add(1);
  CU_TRY(cudaGetLastError());
  CU_TRY(cudaEventRecord(p->blk->ev, st));
  return LIDFE_OK;
}

static int launch_wave(lidfe_handle h, lidfe_plan p, const void* in, int in_i16, float in_scale, float* out, float2* norm_out,
                       int normalize, float dither, const float* noise_dev, float preemph, void* stream) {
  if (!h || !p || !in) return LIDFE_E_NULL;
  if (!out && !norm_out) return LIDFE_E_NULL;
  if (p->ctx != h || in == static_cast<const void*>(out)) return LIDFE_E_ARG;
  WaveParams W = wave_params(p, in, in_i16, in_scale, out, normalize);
  W.norm_out = norm_out;
  W.dither = dither;
  W.noise = noise_dev;
  W.seed = h->cfg.seed;
  W.preemph = preemph;
  return run_wave(p, W, kNoiseNone, stream);
}

// fbank_precise_kernel on the call's parameters: fp64 arithmetic on the same tables, statistics of this launch's parity
static void launch_precise(const lidfe_ctx* h, lidfe_plan p, const FbankParams& P, cudaStream_t st) {
  PreciseParams Q;
  memset(&Q, 0, sizeof(Q));
  Q.wav = P.wav;
  Q.out = P.out;
  Q.out_ld = P.out_ld;
  Q.spans = P.spans;
  Q.n_spans = P.n_spans;
  Q.window = reinterpret_cast<const float*>(h->d_blob);
  Q.mel_k0 = reinterpret_cast<const int*>(h->d_blob + h->k0_off);
  Q.mel_w = reinterpret_cast<const float*>(h->d_blob + h->melw_off);
  for (int b = 0; b < kBands; ++b) Q.band_taps[b] = h->band_taps[b];
  Q.total_taps = h->total_taps;
  Q.dct = h->cfg.n_ceps > 0 ? reinterpret_cast<const float*>(h->d_blob + h->dct_off) : nullptr;
  Q.lifter = h->cfg.n_ceps > 0 ? reinterpret_cast<const float*>(h->d_blob + h->lifter_off) : nullptr;
  Q.n_mels = P.n_mels;
  Q.n_ceps = P.n_ceps;
  Q.n_out = P.n_out;
  Q.preemph = P.preemph;
  Q.in_scale = P.in_scale;
  Q.log_floor = P.log_floor;
  Q.log_of_floor = P.log_of_floor;
  Q.log_mul = (h->cfg.log_kind == LIDFE_LOG_DB10) ? 4.3429448190325182765 : 1.0;     // 10 / ln 10
  Q.center = P.center;
  Q.pad = P.pad;
  Q.utt_offsets = P.utt_offsets;
  Q.utt_lengths = P.utt_lengths;
  Q.utt_max = P.utt_max + static_cast<long long>(P.parity & 1) * P.b_cap;
  Q.utt_min = P.utt_min + static_cast<long long>(P.parity & 1) * P.b_cap;
  Q.remove_dc = P.remove_dc;
  Q.mode = P.mode;
  Q.utt_stats = P.utt_stats + static_cast<long long>(P.parity & 1) * P.b_cap * 2 * h->n_out;
  Q.stats_out = P.stats_out;
  long long gp = p->n_spans * kMaxSpanTiles < static_cast<long long>(h->num_sms) * kPCtasPerSm ? p->n_spans * kMaxSpanTiles : static_cast<long long>(h->num_sms) * kPCtasPerSm;
  if (gp < 1) gp = 1;
  void (*pk)(const PreciseParams) =
      (h->cfg.in_dtype == LIDFE_IN_I16) ? (Q.center ? fbank_precise_kernel<short, true> : fbank_precise_kernel<short, false>)
                                        : (Q.center ? fbank_precise_kernel<float, true> : fbank_precise_kernel<float, false>);
  pk<<<static_cast<unsigned>(gp), kPThreads, kPSmemBytes, st>>>(Q);
}

// The route's feature kernel, bracketed by an event pair between lidfe_profile_begin and lidfe_profile_end (every
// prof_stride-th call).
static int launch_fbank(lidfe_ctx* h, lidfe_plan p, const Route& r, FbankParams& F, cudaStream_t st) {
  bool prof = h->prof_used + 2 <= static_cast<int>(h->prof_events.size());
  if (prof) prof = (h->prof_calls++ % (h->prof_stride > 0 ? h->prof_stride : 1)) == 0;
  if (prof) CU_TRY(cudaEventRecord(h->prof_events[h->prof_used], st));
  if (r.fbank == kFbPrecise) {
    launch_precise(h, p, F, st);
  } else if (r.fbank == kFbWarp) {
    F.wspans = p->d_wspans;
    F.n_wspans = static_cast<int>(p->n_wspans);
    F.w_first = p->d_w_first;
    F.n_wstatic = p->n_wstatic;
    F.w_tab_bytes = h->w_tab_bytes;
    F.const_bytes = h->blob_bytes_fbank;
    long long grid = (p->n_wspans + kWWarps - 1) / kWWarps;      // (never more warps than spans)
    if (grid > h->w_grid || p->n_wstatic > 0) grid = h->w_grid;
    if (grid < 1) grid = 1;
    r.fn<<<static_cast<unsigned>(grid), kWThreads, h->w_smem, st>>>(F);
  } else {
    // the fbank-only variant of the two-kernel MFCC path runs 4 CTAs per SM; a static head of ~85 % of the spans is
    // dealt out as consecutive runs
    const long long cap = r.dct ? static_cast<long long>(h->num_sms) * 4 : h->grid_cap;
    long long grid = p->n_spans < cap ? p->n_spans : cap;
    if (grid < 1) grid = 1;
    const long long ks = ((p->n_spans / grid) * 85) / 100;
    F.k_static = static_cast<int>(ks < 1 ? 1 : ks);
    r.fn<<<static_cast<unsigned>(grid), kThreads, r.dct ? h->smem_bytes_fbank : h->smem_bytes, st>>>(F);
  }
  g_launches.fetch_add(1);
  CU_TRY(cudaGetLastError());
  if (prof) {
    CU_TRY(cudaEventRecord(h->prof_events[h->prof_used + 1], st));
    h->prof_used += 2;
  }
  return LIDFE_OK;
}

// mfcc_dct_mma_kernel: the log-mel workspace's tiles x DCT x lifter into the call's output (P: the call's parameters)
static int launch_dct(const lidfe_ctx* h, lidfe_plan p, const FbankParams& P, cudaStream_t st) {
  DctParams D;
  D.logmel = p->blk->d_logmel;
  D.out = P.out;
  D.out_ld = P.out_ld;
  D.tiles = p->d_tiles;
  D.n_tiles = static_cast<int>(p->n_tiles);
  D.n_mels = h->cfg.n_mels;
  D.n_ceps = h->cfg.n_ceps;
  D.dct = reinterpret_cast<const float*>(h->d_blob + h->dct_off);
  D.lifter = reinterpret_cast<const float*>(h->d_blob + h->lifter_off);
  D.masks = P.masks;
  D.n_masks = P.n_masks;
  D.mode = P.mode;
  D.stats_in = P.stats_in;
  // every warp walks its own contiguous range of tiles; 2 CTAs of 8 warps per SM
  long long gm = (p->n_tiles + kMmTM * kMmWarps - 1) / (kMmTM * kMmWarps);
  if (gm > static_cast<long long>(h->num_sms) * 2) gm = static_cast<long long>(h->num_sms) * 2;
  if (gm < 1) gm = 1;
  mfcc_dct_mma_kernel<<<static_cast<unsigned>(gm), kMmThreads, kMmSmemBytes, st>>>(D);
  g_launches.fetch_add(1);
  CU_TRY(cudaGetLastError());
  return LIDFE_OK;
}

static int featurize_impl(lidfe_handle h, lidfe_plan p, const void* wav_dev, float* out_dev, long long out_ld,
                          const int* masks_dev, int n_masks, int cmvn_mode, const double* stats_in_dev,
                          double* stats_out_dev, void* stream, bool raw) {
  if (!h || !p || !wav_dev || !out_dev) return LIDFE_E_NULL;
  if (p->ctx != h) return LIDFE_E_ARG;
  if (out_ld < h->n_out || cmvn_mode < 0 || cmvn_mode > 4 || n_masks < 0 || n_masks > kMaxMasks) return LIDFE_E_ARG;
  if (cmvn_mode == LIDFE_CMVN_APPLY_GLOBAL && !stats_in_dev) return LIDFE_E_NULL;
  if (cmvn_mode == LIDFE_CMVN_ACCUM_GLOBAL && !stats_out_dev) return LIDFE_E_NULL;
  if (raw && h->precise) return LIDFE_E_ARG;      // the precise kernel has no fused normalize_wav load
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Route r = route_for(h, p, cmvn_mode, raw, masks_dev && n_masks > 0);

  if (raw) {   // statistics pre-pass of normalize_wav: (mean, std + 1e-6) per utterance; the fused kernel applies them
    const int rc = launch_wave(h, p, wav_dev, h->cfg.in_dtype == LIDFE_IN_I16 ? 1 : 0, h->cfg.in_scale, nullptr, p->d_utt_wnorm, 1,
                               0.f, nullptr, 0.f, stream);
    if (rc != LIDFE_OK) return rc;
  }

  FbankParams P;
  memset(&P, 0, sizeof(P));
  P.wav = wav_dev;
  P.out = out_dev;
  P.out_ld = out_ld;
  P.spans = p->d_spans;
  P.n_spans = static_cast<int>(p->n_spans);
  P.sched = p->d_sched;
  P.parity = p->parity;
  P.b_cap = p->blk->Bc;
  if (cmvn_mode == LIDFE_CMVN_PER_UTT || cmvn_mode == LIDFE_POST_TOPDB) p->parity ^= 1;
  P.utt_first_tile = p->d_utt_first_tile;
  P.const_blob = h->d_blob;
  P.const_bytes = h->blob_bytes;
  for (int b = 0; b < kBands; ++b) P.band_taps[b] = h->band_taps[b];
  P.n_mels = h->cfg.n_mels;
  P.n_ceps = h->cfg.n_ceps;
  P.n_out = h->n_out;
  P.preemph = h->cfg.preemph;
  P.log_floor = h->cfg.log_floor;
  if (h->cfg.log_kind == LIDFE_LOG_DB10) {
    P.log_of_floor = 10.0f * log10f(h->cfg.log_floor);       // 10 * log10(amin), fp32 like the reference
    P.log_scale = 3.01029995663981195f;                       // 10 * log10(2)
  } else {
    P.log_of_floor = logf(h->cfg.log_floor);
    P.log_scale = 0.693147180559945309f;                      // ln 2
  }
  P.center = (h->cfg.framing == LIDFE_FRAMING_CENTER) ? 1 : 0;
  P.pad = h->cfg.pad;
  P.utt_offsets = p->d_offsets;
  P.utt_lengths = p->d_lengths;
  P.utt_max = p->d_utt_max;
  P.utt_min = p->d_utt_min;
  P.top_db = h->cfg.top_db;
  P.in_scale = h->cfg.in_scale;
  P.remove_dc = h->cfg.remove_dc;
  P.utt_wnorm = raw ? p->d_utt_wnorm : nullptr;
  P.dither = h->cfg.dither;
  P.seed = h->cfg.seed;
  P.masks = masks_dev;
  P.n_masks = masks_dev ? n_masks : 0;
  P.mode = cmvn_mode;
  P.stats_in = stats_in_dev;
  P.stats_out = stats_out_dev;
  P.utt_stats = p->d_utt_stats;

  FbankParams F = P;
  if (r.dct) {
    // fbank-only: log-mels into the tile-blocked workspace, grown on demand and kept with the pooled block
    PlanBlock* b = p->blk;
    if (b->logmel_tiles < p->n_tiles) {
      CU_TRY(cudaStreamSynchronize(st));
      cudaFree(b->d_logmel);
      b->d_logmel = nullptr;
      b->logmel_tiles = 0;
      const long long cap = pow2_at_least(p->n_tiles, 256);
      CU_TRY(cudaMalloc(reinterpret_cast<void**>(&b->d_logmel), static_cast<size_t>(cap) * kTileFrames * h->cfg.n_mels * sizeof(float)));
      b->logmel_tiles = cap;
    }
    F.out = b->d_logmel;
    F.out_ld = h->cfg.n_mels;
    F.n_ceps = 0;
    F.n_out = h->cfg.n_mels;
    F.masks = nullptr;
    F.n_masks = 0;
    F.mode = LIDFE_CMVN_NONE;
    F.ws_blocked = 1;
    F.const_bytes = h->blob_bytes_fbank;
  }
  int rc = launch_fbank(h, p, r, F, st);
  if (rc == LIDFE_OK && r.dct) rc = launch_dct(h, p, P, st);
  if (rc != LIDFE_OK) return rc;

  if (r.apply == kApplyNone) {
    CU_TRY(cudaEventRecord(p->blk->ev, st));
    return LIDFE_OK;
  }
  const bool parity = r.apply == kApplyUtt || r.apply == kApplyTopDb;
  const int normalize = r.apply == kApplyTopDb ? 2 : r.apply == kApplyMasks ? 0 : 1;
  return launch_apply(h, p, out_dev, out_ld, masks_dev, n_masks, r.apply == kApplyGlobal ? stats_in_dev : nullptr, st,
                      normalize, parity ? P.parity : -1);
}

int lidfe_featurize(lidfe_handle h, lidfe_plan p, const void* wav_dev, float* out_dev, long long out_ld,
                    const int* masks_dev, int n_masks, int cmvn_mode, const double* stats_in_dev,
                    double* stats_out_dev, void* stream) {
  return featurize_impl(h, p, wav_dev, out_dev, out_ld, masks_dev, n_masks, cmvn_mode, stats_in_dev, stats_out_dev, stream, false);
}

int lidfe_featurize_raw(lidfe_handle h, lidfe_plan p, const void* wav_dev, float* out_dev, long long out_ld,
                        const int* masks_dev, int n_masks, int cmvn_mode, const double* stats_in_dev,
                        double* stats_out_dev, void* stream) {
  return featurize_impl(h, p, wav_dev, out_dev, out_ld, masks_dev, n_masks, cmvn_mode, stats_in_dev, stats_out_dev, stream, true);
}

int lidfe_set_precision(lidfe_handle h, int precise) {
  if (!h) return LIDFE_E_NULL;
  if (precise != 0 && precise != 1) return LIDFE_E_ARG;
  if (precise) {
    // scope of fbank_precise_kernel: both framings, both logs; the dither draw stays with the fp32 kernels
    if (h->cfg.dither != 0.f) return LIDFE_E_CONFIG;
    if (h->total_taps > kPMaxTaps) return LIDFE_E_MELBANK;
    cudaError_t e = cudaFuncSetAttribute(fbank_precise_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fbank_precise_kernel<short, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fbank_precise_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fbank_precise_kernel<short, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return static_cast<int>(e);
    }
  }
  h->precise = precise;
  return LIDFE_OK;
}

int lidfe_cmvn_apply(lidfe_handle h, lidfe_plan p, float* feats_dev, long long ld, const int* masks_dev, int n_masks,
                     const double* stats_dev, void* stream) {
  if (!h || !p || !feats_dev || !stats_dev) return LIDFE_E_NULL;
  if (p->ctx != h || ld < h->n_out || n_masks < 0 || n_masks > kMaxMasks) return LIDFE_E_ARG;
  return launch_apply(h, p, feats_dev, ld, masks_dev, n_masks, stats_dev, static_cast<cudaStream_t>(stream), 1);
}

int lidfe_profile_begin(lidfe_handle h, int max_launches) {
  if (!h) return LIDFE_E_NULL;
  if (max_launches <= 0 || !h->prof_events.empty()) return LIDFE_E_ARG;
  try {
    h->prof_events.assign(static_cast<size_t>(max_launches) * 2, nullptr);
  } catch (const std::bad_alloc&) {
    return LIDFE_E_NOMEM;
  }
  h->prof_used = 0;
  h->prof_calls = 0;
  if (h->prof_stride <= 0) h->prof_stride = 1;
  for (auto& ev : h->prof_events) CU_TRY(cudaEventCreate(&ev));
  return LIDFE_OK;
}

int lidfe_profile_set_stride(lidfe_handle h, int stride) {
  if (!h) return LIDFE_E_NULL;
  if (stride < 1) return LIDFE_E_ARG;
  h->prof_stride = stride;
  return LIDFE_OK;
}

int lidfe_profile_end(lidfe_handle h, float* ms_host, int capacity, int* n_out) {
  if (!h || !n_out) return LIDFE_E_NULL;
  if (h->prof_events.empty()) return LIDFE_E_ARG;
  const int n = h->prof_used / 2;
  int rc = LIDFE_OK;
  for (int i = 0; i < n && rc == LIDFE_OK; ++i) {
    cudaError_t e = cudaEventSynchronize(h->prof_events[2 * i + 1]);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, h->prof_events[2 * i], h->prof_events[2 * i + 1]);
    if (e != cudaSuccess) rc = static_cast<int>(e);
    if (ms_host && i < capacity) ms_host[i] = ms;
  }
  for (cudaEvent_t ev : h->prof_events) cudaEventDestroy(ev);
  h->prof_events.clear();
  h->prof_used = 0;
  *n_out = n;
  return rc;
}

int lidfe_mask_apply(lidfe_handle h, lidfe_plan p, float* feats_dev, long long ld, const int* masks_dev, int n_masks,
                     void* stream) {
  if (!h || !p || !feats_dev || !masks_dev) return LIDFE_E_NULL;
  if (p->ctx != h || ld < h->n_out || n_masks < 1 || n_masks > kMaxMasks) return LIDFE_E_ARG;
  return launch_apply(h, p, feats_dev, ld, masks_dev, n_masks, nullptr, static_cast<cudaStream_t>(stream), 0);
}

int lidfe_wave_stages(lidfe_handle h, lidfe_plan p, const float* wav_in_dev, float* wav_out_dev, int normalize,
                      float dither, const float* noise_dev, float preemph, void* stream) {
  if (!wav_out_dev) return LIDFE_E_NULL;
  return launch_wave(h, p, wav_in_dev, 0, 1.f, wav_out_dev, nullptr, normalize, dither, noise_dev, preemph, stream);
}

int lidfe_wave_stages_i16(lidfe_handle h, lidfe_plan p, const short* pcm_in_dev, float in_scale, float* wav_out_dev,
                          int normalize, float dither, const float* noise_dev, float preemph, void* stream) {
  if (!wav_out_dev) return LIDFE_E_NULL;
  return launch_wave(h, p, pcm_in_dev, 1, in_scale, wav_out_dev, nullptr, normalize, dither, noise_dev, preemph, stream);
}

int lidfe_add_noise(lidfe_handle h, lidfe_plan p, const void* wav_in_dev, int in_i16, float in_scale, float* wav_out_dev,
                    const float* bank_dev, long long bank_len, const long long* noise_tab_dev, const float* snr_db_dev,
                    unsigned long long seed, int normalize, void* stream) {
  if (!h || !p || !wav_in_dev || !wav_out_dev || !snr_db_dev) return LIDFE_E_NULL;
  if (bank_dev && !noise_tab_dev) return LIDFE_E_NULL;
  if (p->ctx != h || wav_in_dev == static_cast<const void*>(wav_out_dev) || (in_i16 != 0 && in_i16 != 1)) return LIDFE_E_ARG;
  if (bank_dev && (bank_len <= 0 || bank_dev == wav_out_dev)) return LIDFE_E_ARG;
  WaveParams W = wave_params(p, wav_in_dev, in_i16, in_scale, wav_out_dev, normalize ? 1 : 0);
  W.bank = bank_dev;
  W.bank_len = bank_len;
  W.noise_tab = noise_tab_dev;
  W.snr_db = snr_db_dev;
  W.noise_seed = seed;
  return run_wave(p, W, bank_dev ? kNoiseBank : kNoiseGauss, stream);
}

// ---- FP32 ceiling, measured (bench.py's roofline denominator) -----------------------------------------------------
__global__ void __launch_bounds__(256) fp32_probe_kernel(float* out, float seed, int iters) {
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = seed + i + threadIdx.x;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = fmaf(a[i], seed, 0.5f);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += a[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

int lidfe_fp32_probe(float ms_budget, double* tflops_out, void* stream) {
  if (!tflops_out) return LIDFE_E_NULL;
  if (!(ms_budget > 0.f)) return LIDFE_E_ARG;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int dev = 0, sms = 0;
  CU_TRY(cudaGetDevice(&dev));
  CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int threads = 256, blocks = sms * 8, iters = 4096;
  float* out = nullptr;
  CU_TRY(cudaMalloc(reinterpret_cast<void**>(&out), sizeof(float) * threads * blocks));
  cudaEvent_t e0, e1;
  CU_TRY(cudaEventCreate(&e0));
  CU_TRY(cudaEventCreate(&e1));
  fp32_probe_kernel<<<blocks, threads, 0, st>>>(out, 1.0001f, iters);     // warm-up
  double best = 0.0;
  float spent = 0.f;
  cudaError_t e = cudaSuccess;
  for (int r = 0; r < 64 && spent < ms_budget && e == cudaSuccess; ++r) {
    cudaEventRecord(e0, st);
    fp32_probe_kernel<<<blocks, threads, 0, st>>>(out, 1.0001f, iters);
    cudaEventRecord(e1, st);
    e = cudaEventSynchronize(e1);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    g_launches.fetch_add(1);
    spent += ms;
    if (ms > 0.f) {
      const double tf = 2.0 * 8.0 * iters * static_cast<double>(threads) * blocks / (ms * 1e-3) / 1e12;
      best = tf > best ? tf : best;
    }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return static_cast<int>(e);
  }
  *tflops_out = best;
  return LIDFE_OK;
}

// ---- polyphase sinc resampler (row f4) ---------------------------------------------------------------------------
struct lidfe_resampler_s {
  int orig, nw, K, K4, width;      // frequencies already divided by their gcd
  float* d_wt;                     // [K4][nw] transposed bank (FP32 kernel)
  // tcgen05 path (lidfe_resample_tc.cuh): the bank as shared-memory images, one per (phase tile, 32-tap block, hi | lo)
  int use_tc, tc_N, tc_tiles, tc_KB, tc_stages, tc_cols;
  size_t tc_smem;
  unsigned char* d_wimg;
};

// fp32 -> tf32, round to nearest with ties away from zero (what cvt.rna.tf32.f32 does), on the host
static float tf32_rna_host(float v) {
  uint32_t u;
  memcpy(&u, &v, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return v;         // inf / nan
  u += 0x1000u;
  u &= 0xffffe000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

static int create_bank(lidfe_resampler* out, int orig, int nw, const float* kernel_host, int taps, int width);

int lidfe_resampler_create(lidfe_resampler* out, int orig_freq, int new_freq, const float* kernel_host, int taps, int width) {
  if (!out || !kernel_host) return LIDFE_E_NULL;
  *out = nullptr;
  if (orig_freq <= 0 || new_freq <= 0 || taps <= 0 || width < 0 || taps > 8192) return LIDFE_E_ARG;
  int a = orig_freq, b = new_freq;
  while (b) { const int t = a % b; a = b; b = t; }
  const int orig = orig_freq / a, nw = new_freq / a;
  if (taps != 2 * width + orig) return LIDFE_E_ARG;     // ta: functional/functional.py _get_sinc_resample_kernel
  return create_bank(out, orig, nw, kernel_host, taps, width);
}

// The resampler kernels are a windowed GEMM -- out[f * n_rows + p] = sum_k bank[p][k] * xpad[f * hop - left_pad + k] --
// and any bank can be run through them: the wav2vec-exp FBank variant uses a windowed DFT basis (lidfe_stft_fbank.cuh).
int lidfe_wgemm_create(lidfe_resampler* out, int hop, int n_rows, const float* bank_host, int taps, int left_pad) {
  if (!out || !bank_host) return LIDFE_E_NULL;
  *out = nullptr;
  if (hop <= 0 || n_rows <= 0 || taps <= 0 || left_pad < 0 || taps > 8192 || (n_rows & 1)) return LIDFE_E_ARG;
  return create_bank(out, hop, n_rows, bank_host, taps, left_pad);
}

static int create_bank(lidfe_resampler* out, int orig, int nw, const float* kernel_host, int taps, int width) {
  lidfe_resampler_s* r = new (std::nothrow) lidfe_resampler_s();
  if (!r) return LIDFE_E_NOMEM;
  r->orig = orig; r->nw = nw; r->K = taps; r->K4 = (taps + 3) & ~3; r->width = width; r->d_wt = nullptr;
  std::vector<float> wt(static_cast<size_t>(r->K4) * nw, 0.f);
  for (int p = 0; p < nw; ++p)
    for (int k = 0; k < taps; ++k) wt[static_cast<size_t>(k) * nw + p] = kernel_host[static_cast<size_t>(p) * taps + k];
  cudaError_t e = upload(&r->d_wt, wt.data(), wt.size());
  const size_t smem = static_cast<size_t>(kRsFrames) * r->K4 * sizeof(float);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  // tcgen05 path: phases in tiles of N, the largest multiple of 32 that divides nw and is <= 256 (160 for both of the
  // reference's rates), else the largest such multiple of 16 (M = 128 takes any N % 16 == 0 up to 256)
  r->use_tc = 0;
  r->d_wimg = nullptr;
  {
    int N = 0;
    for (int c = 256; c >= 32 && N == 0; c -= 32)
      if (nw % c == 0) N = c;
    for (int c = 240; c >= 16 && N == 0; c -= 16)
      if (nw % c == 0) N = c;
    // test selector: LIDFE_RESAMPLE_TC=0 keeps resample_kernel, the FP32 reference the tensor-core kernel is tested against
    const char* et = getenv("LIDFE_RESAMPLE_TC");
    int dev = 0, cc_major = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e == cudaSuccess && N > 0 && cc_major == 10 && !(et && et[0] == '0')) {
      r->tc_N = N;
      r->tc_tiles = nw / N;
      r->tc_KB = (taps + kTcKB - 1) / kTcKB;
      if (r->tc_KB < 2) r->tc_KB = 2;                         // the builder warps' two sets: a second block of zeros
      const size_t stage = 2 * static_cast<size_t>(kTcABytes) + 2 * static_cast<size_t>(N) * 128;
      int stages = static_cast<int>((220 * 1024) / stage);    // >= 2: a stage is at most 96 KB (N <= 256)
      if (stages > 4) stages = 4;
      if (stages > r->tc_KB) stages = r->tc_KB;
      r->tc_stages = stages;
      // two accumulator buffers of tc_cols / 2 >= round_up(N, 32) columns each: the epilogue reads 32 columns at a time
      r->tc_cols = 32;
      while (r->tc_cols < 2 * ((N + 31) & ~31)) r->tc_cols <<= 1;
      r->tc_smem = stages * stage + 1024 + (3 * static_cast<size_t>(stages) + 5) * 8;
      // image of (tile t, block kb, part h): row n (phase t N + n) holds taps 32 kb .. 32 kb + 31 in 128 bytes, its eight
      // 16-byte chunks XOR-swizzled by n % 8 (the layout tcgen05.mma reads with a SWIZZLE_128B K-major descriptor)
      const size_t img = static_cast<size_t>(N) * 128;
      std::vector<float> buf(static_cast<size_t>(r->tc_tiles) * r->tc_KB * 2 * (img / 4), 0.f);
      for (int t = 0; t < r->tc_tiles; ++t)
        for (int kb = 0; kb < r->tc_KB; ++kb)
          for (int n = 0; n < N; ++n)
            for (int kk = 0; kk < kTcKB; ++kk) {
              const int k = kb * kTcKB + kk;
              const float w = (k < taps) ? kernel_host[static_cast<size_t>(t * N + n) * taps + k] : 0.f;
              const float hi = tf32_rna_host(w), lo = w - hi;
              const size_t off = (static_cast<size_t>(n) * 128 + ((((kk >> 2) ^ (n & 7)) << 4) | ((kk & 3) << 2))) / 4;
              const size_t base = (static_cast<size_t>(t) * r->tc_KB + kb) * 2 * (img / 4);
              buf[base + off] = hi;
              buf[base + img / 4 + off] = lo;
            }
      float* dimg = nullptr;
      e = upload(&dimg, buf.data(), buf.size());
      r->d_wimg = reinterpret_cast<unsigned char*>(dimg);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(resample_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(r->tc_smem));
      r->use_tc = (e == cudaSuccess);
    }
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    cudaFree(r->d_wt);
    cudaFree(r->d_wimg);
    delete r;
    return static_cast<int>(e);
  }
  *out = r;
  return LIDFE_OK;
}

int lidfe_resampler_destroy(lidfe_resampler r) {
  if (!r) return LIDFE_E_NULL;
  cudaFree(r->d_wt);
  cudaFree(r->d_wimg);
  delete r;
  return LIDFE_OK;
}

long long lidfe_resample_out_len(lidfe_resampler r, long long n_in) {
  if (!r || n_in < 0) return 0;
  return (static_cast<long long>(r->nw) * n_in + r->orig - 1) / r->orig;      // ceil(new * n / orig)
}

int lidfe_resample(lidfe_resampler r, int B, const float* in_dev, const long long* in_off_dev, const long long* in_len_dev,
                   float* out_dev, const long long* out_off_dev, const long long* out_len_dev, long long max_out_len,
                   void* stream) {
  if (!r || !in_dev || !in_off_dev || !in_len_dev || !out_dev || !out_off_dev || !out_len_dev) return LIDFE_E_NULL;
  if (B <= 0 || max_out_len < 0) return LIDFE_E_ARG;
  if (max_out_len == 0) return LIDFE_OK;
  if (r->use_tc) {
    ResampleTcParams T;
    T.in = in_dev; T.in_off = in_off_dev; T.in_len = in_len_dev;
    T.out = out_dev; T.out_off = out_off_dev; T.out_len = out_len_dev;
    T.wimg = r->d_wimg; T.orig = r->orig; T.nw = r->nw; T.K = r->K; T.KB = r->tc_KB; T.width = r->width;
    T.N = r->tc_N; T.stages = r->tc_stages; T.tmem_cols = r->tc_cols;
    const long long fr = (max_out_len + r->nw - 1) / r->nw;
    const long long gxt = (fr + kTcM - 1) / kTcM;
    if (gxt > 0x7fffffffLL || B > 65535 || r->tc_tiles > 65535) return LIDFE_E_ARG;
    T.gx = static_cast<int>(gxt); T.B = B; T.n_tiles = r->tc_tiles;
    const long long n_lin = gxt * B * r->tc_tiles;
    int dev = 0, sms = 0;
    CU_TRY(cudaGetDevice(&dev));
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const long long grid = n_lin < sms ? n_lin : sms;         // persistent: one CTA per SM walks the tiles
    resample_tc_kernel<<<static_cast<unsigned>(grid), kTcThreads, r->tc_smem, static_cast<cudaStream_t>(stream)>>>(T);
    g_launches.fetch_add(1);
    CU_TRY(cudaGetLastError());
    return LIDFE_OK;
  }
  ResampleParams P;
  P.in = in_dev; P.in_off = in_off_dev; P.in_len = in_len_dev;
  P.out = out_dev; P.out_off = out_off_dev; P.out_len = out_len_dev;
  P.wt = r->d_wt; P.orig = r->orig; P.nw = r->nw; P.K = r->K; P.K4 = r->K4; P.width = r->width;
  const long long frames = (max_out_len + r->nw - 1) / r->nw;
  const long long gx = (frames + kRsFrames - 1) / kRsFrames;
  if (gx > 0x7fffffffLL || B > 65535) return LIDFE_E_ARG;
  const size_t smem = static_cast<size_t>(kRsFrames) * r->K4 * sizeof(float);
  resample_kernel<<<dim3(static_cast<unsigned>(gx), static_cast<unsigned>(B)), kRsThreads, smem, static_cast<cudaStream_t>(stream)>>>(P);
  g_launches.fetch_add(1);
  CU_TRY(cudaGetLastError());
  return LIDFE_OK;
}

}  // extern "C"
