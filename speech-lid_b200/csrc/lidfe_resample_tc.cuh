// lidfe_resample_tc.cuh -- the polyphase resampler GEMM on the 5th-generation tensor cores (tcgen05 + TMEM), row f4.
//
// out[frame * nw + p] = sum_k W[p][k] * xpad[frame * orig - width + k]        (ref: lid/ConformerLangModel.py:131-178 ->
// ta: functional/functional.py _apply_sinc_resample_kernel: a strided conv1d = a GEMM whose left operand is an im2col
// view of the waveform).  One CTA computes 128 consecutive frames of one utterance for N phases:
//   D[128 frames x N phases] (fp32, in TMEM) = A[128 x K] . B[N x K]^T,  both operands K-major in shared memory,
// as 3 x TF32: every fp32 value is split once into hi = tf32(v) and lo = v - hi, and D += A_lo.B_hi + A_hi.B_lo + A_hi.B_hi
// (the product of the two low parts is below fp32 resolution), to the 1e-5 parity bar of the FP32 resample_kernel, with
// tcgen05.mma issued by one thread, accumulators in tensor memory, and the operands staged through a 3-stage mbarrier
// pipeline:
//   * B (the FIR bank) is constant: the host lays every (phase tile, 32-tap block) out as the exact shared-memory image
//     -- rows of 128 bytes, 16-byte chunks XOR-swizzled by (row % 8), hi image then lo image -- so one 1-D TMA bulk copy
//     (cp.async.bulk, complete_tx on the stage's mbarrier) brings a block in;
//   * A cannot come by TMA: its rows are windows of the waveform `orig` samples apart (441 * 4 bytes is no multiple of 16),
//     so four builder warps gather them -- one coalesced 128-byte load per row and block, split, two conflict-free
//     STS.32 into the same swizzled layout -- and publish the stage with fence.proxy.async + mbarrier arrive;
//   * one lane of the MMA warp waits for both, issues 4 k-steps x 3 tcgen05.mma (M 128, N, K 8) per block and hands the
//     stage back with tcgen05.commit; a last commit tells the builder warps, which double as the epilogue, that the
//     accumulators are complete: tcgen05.ld (32 lanes x 32 columns per warp and turn) -> registers -> global.
// SASS of this kernel: UTCHMMA / UTCBAR / LDTM / UBLKCP (profiles/r2_resample_tc_sass.txt).
// Scope: nw % 16 == 0, any number of taps (fewer than 33 run as two blocks, the second all zeros); resample_kernel takes
// every other rate pair.
#pragma once
#include "lidfe_kernels.cuh"

namespace lidfe {

constexpr int kTcM = 128;            // frames per CTA = rows of A = TMEM lanes
constexpr int kTcKB = 32;            // taps per pipeline stage = one 128-byte swizzle row
constexpr int kTcThreads = 512;      // warp 0: B loader, 1: MMA issuer + TMEM owner, 4-11: A builders, 12-15: epilogue
constexpr int kTcABytes = kTcM * kTcKB * 4;          // 16 KB per (hi | lo) image of A

struct ResampleTcParams {
  const float* in;
  const long long* in_off;
  const long long* in_len;
  float* out;
  const long long* out_off;
  const long long* out_len;
  const unsigned char* wimg;         // [n_tiles][KB][2][N * 128 bytes] shared-memory images of the FIR bank (hi, lo)
  int orig, nw, K, KB, width;        // KB = max(2, ceil(K / 32)) tap blocks
  int N, stages, tmem_cols;          // phases per CTA (multiple of 16, <= 256), pipeline depth, allocated TMEM columns (2 buffers)
  int gx, B, n_tiles;                // tile grid: frame tiles per utterance (of the longest), utterances, phase tiles
};

template <bool kRelaxed = false>
__device__ __forceinline__ void tc_wait(uint64_t* bar, uint32_t parity) {
  // bounded: a descriptor mistake must end in a trap the host sees, not in a hung GPU.  kRelaxed: waiters off the critical
  // path (B loader, epilogue) back off between polls so that their spinning does not take issue slots from the builders
  for (uint32_t spins = 0;; ++spins) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) return;
    if (kRelaxed) __nanosleep(128);
    if (spins > (1u << 24)) __trap();
  }
}

// shared-memory matrix descriptor, K-major, 128-byte swizzle: rows of 128 bytes, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu);      // start address
  d |= static_cast<uint64_t>(1u) << 16;                        // leading byte offset (unused with swizzle): 1
  d |= static_cast<uint64_t>(1024u >> 4) << 32;                // stride byte offset: next 8-row group
  d |= static_cast<uint64_t>(1u) << 46;                        // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2u) << 61;                        // SWIZZLE_128B
  return d;
}

__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(kTcThreads, 1) resample_tc_kernel(const __grid_constant__ ResampleTcParams P) {
  extern __shared__ unsigned char tc_smem_raw[];
  // 1024-byte aligned stage buffers (the swizzle works on absolute shared-memory address bits)
  unsigned char* const base = tc_smem_raw + ((1024u - (smem_u32(tc_smem_raw) & 1023u)) & 1023u);
  const int b_bytes = P.N * 128;                                   // one (hi | lo) image of B
  const int stage_bytes = 2 * kTcABytes + 2 * b_bytes;
  uint64_t* const bars = reinterpret_cast<uint64_t*>(base + P.stages * stage_bytes);
  uint64_t* const full_a = bars;                                   // [stages] 4 builder warps
  uint64_t* const full_b = bars + P.stages;                        // [stages] TMA bytes
  uint64_t* const empty = bars + 2 * P.stages;                     // [stages] tcgen05.commit
  uint64_t* const acc_full = bars + 3 * P.stages;                  // [2] accumulators of a tile complete (tcgen05.commit)
  uint64_t* const acc_empty = bars + 3 * P.stages + 2;             // [2] ... and read out by the four epilogue warps
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * P.stages + 4);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full_a[s], 4);                                    // one arrival per builder warp of the item's set
      mbar_init(&full_b[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&acc_full[a], 1);
      mbar_init(&acc_empty[a], 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {                                                 // TMEM: allocated and later freed by this warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(static_cast<uint32_t>(P.tmem_cols)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  const uint32_t acc_stride = static_cast<uint32_t>(P.tmem_cols >> 1);   // two accumulator buffers

  // Persistent CTA: tiles blockIdx.x, blockIdx.x + gridDim.x, ... of the (frame tile, utterance, phase tile) grid; tiles
  // past an utterance's end are skipped by every role alike.  `seq` counts the tiles a CTA has worked on: tap block kb of
  // tile seq is pipeline item seq * KB + kb (stage = item % stages), its accumulators live in buffer seq & 1.
  const long long n_lin = static_cast<long long>(P.gx) * P.B * P.n_tiles;
  auto tile_live = [&](long long L, int& bb, int& nt, long long& f0) -> bool {
    bb = static_cast<int>((L / P.gx) % P.B);
    nt = static_cast<int>(L / (static_cast<long long>(P.gx) * P.B));
    f0 = (L % P.gx) * kTcM;
    return f0 * P.nw < P.out_len[bb];
  };
  auto next_live = [&](long long L) -> long long {                  // first live tile of this CTA at or after L
    int bb, nt; long long f0;
    while (L < n_lin && !tile_live(L, bb, nt, f0)) L += gridDim.x;
    return L;
  };

  if (warp == 0) {
    // ---- B loader: one bulk copy per tap block (hi and lo images are adjacent in the host-built table) -------------
    if (lane == 0) {
      uint32_t item = 0;
      for (long long L = next_live(blockIdx.x); L < n_lin; L = next_live(L + gridDim.x)) {
        int bb, nt; long long f0;
        tile_live(L, bb, nt, f0);
        const unsigned char* src = P.wimg + static_cast<long long>(nt) * P.KB * 2 * b_bytes;
        for (int kb = 0; kb < P.KB; ++kb, ++item) {
          const uint32_t s = item % P.stages, u = item / P.stages;
          if (u > 0) tc_wait<true>(&empty[s], (u - 1) & 1u);
          mbar_expect_tx(&full_b[s], static_cast<uint32_t>(2 * b_bytes));
          tma_bulk_g2s_plain(base + s * stage_bytes + 2 * kTcABytes, src + static_cast<long long>(kb) * 2 * b_bytes,
                             static_cast<uint32_t>(2 * b_bytes), &full_b[s]);
        }
      }
    }
  } else if (warp == 1) {
    // ---- MMA issuer: one lane ------------------------------------------------------------------------------------
    if (lane == 0) {
      // instruction descriptor: D fp32, A and B tf32, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(P.N >> 3) << 17) |
                             (static_cast<uint32_t>(kTcM >> 4) << 24);
      uint32_t item = 0, seq = 0;
      for (long long L = next_live(blockIdx.x); L < n_lin; L = next_live(L + gridDim.x), ++seq) {
        const uint32_t a = seq & 1u;
        if (seq >= 2) {                                            // the epilogue has drained this buffer's previous tile
          tc_wait(&acc_empty[a], ((seq >> 1) - 1) & 1u);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        const uint32_t d_addr = tmem_d + a * acc_stride;
        for (int kb = 0; kb < P.KB; ++kb, ++item) {
          const uint32_t s = item % P.stages, u = item / P.stages;
          tc_wait(&full_a[s], u & 1u);
          tc_wait(&full_b[s], u & 1u);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_hi = smem_u32(base + s * stage_bytes), a_lo = a_hi + kTcABytes;
          const uint32_t b_hi = a_hi + 2 * kTcABytes, b_lo = b_hi + b_bytes;
#pragma unroll
          for (int j = 0; j < kTcKB / 8; ++j) {                    // K = 8 tf32 = 32 bytes per instruction
            const uint32_t off = 32u * j;
            tc_mma_tf32(d_addr, tc_smem_desc(a_lo + off), tc_smem_desc(b_hi + off), idesc, (kb | j) ? 1u : 0u);
            tc_mma_tf32(d_addr, tc_smem_desc(a_hi + off), tc_smem_desc(b_lo + off), idesc, 1u);
            tc_mma_tf32(d_addr, tc_smem_desc(a_hi + off), tc_smem_desc(b_hi + off), idesc, 1u);
          }
          tc_commit(&empty[s]);                                    // the stage is free once these MMAs have read it
        }
        tc_commit(&acc_full[a]);
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ---- A builders: warps 4-7 take the even pipeline items, warps 8-11 the odd ones; warp (set, q) gathers rows
    //      32 q .. 32 q + 31 of its items, with the loads of its next item in flight while it stores the current one
    //      (one block at a time, the L2 round trip of the gather -- not the MMA -- paced the tile) ----------------------
    const int q = (warp - 4) & 3, set = (warp - 4) >> 2;
    struct Pos { long long L, f0, n_in; const float* x; int kb; uint32_t item; };
    auto load_tile = [&](Pos& p) {
      if (p.L >= n_lin) return;
      int bb, nt;
      tile_live(p.L, bb, nt, p.f0);
      p.n_in = P.in_len[bb];
      p.x = P.in + P.in_off[bb];
    };
    auto advance2 = [&](Pos& p) {                                  // two items on (the other set takes the one in between)
      p.kb += 2;
      p.item += 2;
      bool moved = false;
      while (p.kb >= P.KB && p.L < n_lin) {
        p.kb -= P.KB;
        p.L = next_live(p.L + gridDim.x);
        moved = true;
      }
      if (moved) load_tile(p);
    };
    // (the builders' instruction stream, not memory or the tensor core, paces the pipeline -- with loads, MMAs and B copies
    //  all ablated a tile still took 17 of 26 us -- so a block that lies inside the utterance takes a path without any
    //  per-element index arithmetic or bounds test: one multiply-add for the address, cvt + sub + xor + 2 stores to publish)
    auto gather = [&](const Pos& p, float (&v)[32]) {
      const int k = p.kb * kTcKB + lane;                           // this lane's tap
      const long long j0 = (p.f0 + 32 * q) * P.orig - P.width + k; // sample of row 32 q at this tap
      const float* const src = p.x + j0;
      if (j0 >= 0 && j0 + 31ll * P.orig < p.n_in && p.kb * kTcKB + 31 < P.K) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __ldg(src + i * P.orig);
        // a row moves on by one 128-byte line per tap block: ask L2 for the line this warp's NEXT-BUT-ONE block will
        // touch (its own next block is already being loaded into the other register buffer) -- the builders' exposed
        // DRAM latency was 40 % of the tile (clock64 cycle counters)
        if (lane == 0 && j0 + 31ll * P.orig + 5 * kTcKB < p.n_in) {
#pragma unroll
          for (int i = 0; i < 32; ++i) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + i * P.orig + 4 * kTcKB + 31));
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const long long j = j0 + static_cast<long long>(i) * P.orig;
          v[i] = (k < P.K && j >= 0 && j < p.n_in) ? __ldg(p.x + j) : 0.f;
        }
      }
    };
    const uint32_t a_lane = static_cast<uint32_t>(32 * q * 128 + ((lane & 3) << 2));   // row 32 q, this lane's word in a chunk
    const uint32_t chunk = static_cast<uint32_t>(lane >> 2);
    auto publish = [&](uint32_t item, const float (&v)[32]) {
      const uint32_t s = item % P.stages, u = item / P.stages;
      if (u > 0) tc_wait(&empty[s], (u - 1) & 1u);
      const uint32_t a_hi = smem_u32(base + s * stage_bytes) + a_lane;
#pragma unroll
      for (int i = 0; i < 32; ++i) {                               // row 32 q + i: chunk c goes to position c ^ (row % 8)
        uint32_t hi, lo;
        split_tf32(v[i], hi, lo);
        const uint32_t addr = a_hi + static_cast<uint32_t>(i * 128) + ((chunk ^ static_cast<uint32_t>(i & 7)) << 4);
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(hi) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr + kTcABytes), "r"(lo) : "memory");
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(&full_a[s]);                      // (128 arrivals on one mbarrier cost 0.26 us per item)
    };
    Pos p;
    p.L = next_live(blockIdx.x);
    p.kb = set - 2;
    p.item = static_cast<uint32_t>(set - 2);
    p.f0 = 0; p.n_in = 0; p.x = P.in;
    load_tile(p);
    advance2(p);                                                   // -> this set's first item (kb = set; KB >= 2)
    float va[32], vb[32];
    if (p.L < n_lin) gather(p, va);
    while (p.L < n_lin) {
      const uint32_t ia = p.item;
      advance2(p);
      const bool have_b = p.L < n_lin;
      const uint32_t ib = p.item;
      if (have_b) gather(p, vb);
      publish(ia, va);
      if (!have_b) break;
      advance2(p);
      if (p.L < n_lin) gather(p, va);
      publish(ib, vb);
    }
  } else if (warp >= 12) {
    // ---- epilogue: TMEM lane = frame, column = phase; the buffer goes back to the MMA warp as soon as it is in registers --
    const int q = warp - 12;
    uint32_t seq = 0;
    for (long long L = next_live(blockIdx.x); L < n_lin; L = next_live(L + gridDim.x), ++seq) {
      int bb, nt; long long f0;
      tile_live(L, bb, nt, f0);
      const long long n_out = P.out_len[bb];
      const uint32_t a = seq & 1u;
      tc_wait<true>(&acc_full[a], (seq >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      float* const y = P.out + P.out_off[bb];
      const long long o_row = (f0 + 32 * q + lane) * P.nw + static_cast<long long>(nt) * P.N;
      for (int c = 0; c < P.N; c += 32) {                           // (a buffer is at least round_up(N, 32) columns wide)
        uint32_t r[32];
        const uint32_t taddr = tmem_d + a * acc_stride + (static_cast<uint32_t>(32 * q) << 16) + static_cast<uint32_t>(c);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
              "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
              "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
              "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (c + 32 >= P.N) {                                       // last chunk read: hand the buffer back before the stores
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[a]);
        }
        const long long o = o_row + c;
        const int nv = P.N - c < 32 ? P.N - c : 32;                // valid columns of this chunk
        if (nv == 32 && o + 32 <= n_out && ((reinterpret_cast<uintptr_t>(y + o) & 15) == 0)) {
#pragma unroll
          for (int e = 0; e < 32; e += 4)
            *reinterpret_cast<float4*>(y + o + e) = make_float4(__uint_as_float(r[e]), __uint_as_float(r[e + 1]),
                                                                __uint_as_float(r[e + 2]), __uint_as_float(r[e + 3]));
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (e < nv && o + e < n_out) y[o + e] = __uint_as_float(r[e]);
        }
      }
    }
  }

  // ---- teardown: every tcgen05 operation of this CTA is complete before the columns go back ------------------------
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(static_cast<uint32_t>(P.tmem_cols)) : "memory");
  }
}

}  // namespace lidfe
