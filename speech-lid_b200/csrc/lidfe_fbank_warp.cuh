// lidfe_fbank_warp.cuh -- the warp-autonomous flavour of the fused front-end kernel (round 2).
//
// Same arithmetic as fbank_kernel (lidfe_kernels.cuh: frame-pair packed f32x2, 16 x 16 FFT, segment-form mel), other
// control structure.  ncu's per-instruction stall samples of the CTA-tiled kernel (profiles/r2_stall_profile.txt) put
// ~40 % of the warp time OUTSIDE the arithmetic: waiting on the CTA-shared sample buffer's mbarrier (the next tile's TMA
// copy could only be issued once the slowest of the 4 warps had consumed the current one), CTA barriers at every span
// end, the shared arrival counter, and the fp64 statistics pass through shared memory.  Here every WARP is a worker of
// its own:
//   * work unit = a QUAD of 4 consecutive frames of one utterance (two frame pairs, one per half-warp); a warp walks
//     "warp spans" (runs of quads of one utterance), first a static run of consecutive spans, then spans claimed one
//     at a time from a global counter (claimed two spans ahead, descriptor fetched by cp.async one span ahead);
//   * each warp owns a private 880-sample staging buffer and mbarrier.  The warp copies the quad's samples into
//     registers (18 LDS.64 per lane, ~10 % into the quad) and at once issues the TMA bulk copy of its NEXT quad -- also
//     across span boundaries -- which lands under the remaining ~90 %.  Nothing in the steady state synchronises two
//     warps: no CTA barrier, no shared counter.  (The 240-sample halo of a quad is fetched again by the warp that owns
//     the next quad: 1.375 x L2 -> SM traffic, HBM traffic unchanged, the halo is in L2.)
//   * ONE transposition between the two FFT stages: (re_A, re_B, im_A, im_B) of a point travel together as one 16-byte
//     element (STS.128 / LDS.128, row stride 17 elements: conflict free both ways).  A point's registers are dead as soon
//     as it has been stored, which lets the compiler load the next twiddles ahead of their use; two warp barriers per
//     quad instead of four.
//   * statistics (per-utterance / global CMVN sums) stay in registers as CENTRED fp32 partial sums of a few quads and
//     are folded into lane-owned fp64 accumulators in the warp's shared memory every kFoldQuads quads; they leave the
//     warp with fp64 atomics when the utterance changes (per-utterance mode) or once per CTA at the end (global mode).
//     The statistics-free instantiation (kStats = false) carries none of those registers.
// Scope: KALDI framing (kStdMel 0 / 1) and the reference's default branch -- CENTER framing, HTK mel, 10 log10, per-utterance
// extrema for AmplitudeToDB(top_db) (kStdMel 2) --, 16-byte aligned utterances, cmvn modes none / per-utterance statistics /
// global apply / global accumulate / top_db, fbank output (the MFCC two-kernel path uses it with the tile-blocked workspace
// layout).  Everything else (in-kernel dither / normalize_wav, in-kernel DCT, unaligned offsets, generic CENTER configs) stays
// with fbank_kernel.
#pragma once
#include "lidfe_kernels.cuh"

namespace lidfe {

constexpr int kQuadFrames = 4;
constexpr int kQuadSamples = kFrameShift * kQuadFrames + (kFrameLen - kFrameShift);   // 880
constexpr int kWWarps = 16;                      // warps per CTA (they only share the constant tables)
constexpr int kWCtasPerSm = 1;
constexpr int kWThreads = kWWarps * 32;
constexpr int kFoldQuads = 32;                   // fp32 partial sums are folded into the fp64 accumulators this often
constexpr int kWTabOff = 128;                    // tables start here (the tables' mbarrier sits in front)

// per half-warp transposition plane: 16 rows of 17 elements of 16 bytes (re_A, re_B, im_A, im_B); reused for the 257
// power pairs of the mel stage
constexpr int kXRow = 17;                        // float4 elements per row
constexpr int kXPlaneBytes = 16 * kXRow * 16;    // 4352

template <typename TIn>
struct WarpLayout {
  static constexpr int kInBytes = (kQuadSamples * static_cast<int>(sizeof(TIn)) + 15) / 16 * 16;   // 3520 (f32) / 1760 (i16)
  static constexpr int off_in = 0;
  static constexpr int off_plane = kInBytes;                       // two half-warp planes
  static constexpr int off_aux = off_plane + 2 * kXPlaneBytes;     // kStats: 80 + 80 fp64 accumulators; else the mask table
  static constexpr int off_ctl = off_aux + 2 * kMaxMels * 8;       // mbarrier @0 | span slots @16, @48 (32 B each)
  static constexpr int kWarpBytes = off_ctl + 80;
};

struct WSpanRegs {     // the fields of a span a warp needs per quad, read from its shared-memory slot when needed
  long long wav_off, out_row;
  int nframes, utt, t0, aux;
};

// kStats: 0 = no statistics, 1 = sums for per-utterance / global CMVN, 2 = per-utterance extrema for AmplitudeToDB(top_db)
template <typename TIn, int kStdMel, int kStats>
__global__ void __launch_bounds__(kWThreads, kWCtasPerSm) fbank_warp_kernel(const __grid_constant__ FbankParams P) {
  using L0 = SmemLayout<float, false>;
  using WL = WarpLayout<TIn>;
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* const tab_bar = reinterpret_cast<uint64_t*>(smem);
  unsigned char* const tab = smem + kWTabOff;
  const float* const sm_window = reinterpret_cast<const float*>(tab);
  const float2* const sm_tw1 = reinterpret_cast<const float2*>(tab + (L0::off_tw1 - L0::off_window));
  const float2* const sm_tw2 = reinterpret_cast<const float2*>(tab + (L0::off_tw2 - L0::off_window));
  const int* const sm_k0 = reinterpret_cast<const int*>(tab + (L0::off_k0 - L0::off_window));
  const float* const sm_melw = reinterpret_cast<const float*>(tab + (L0::off_melw - L0::off_window));
  float2* const sm_norm = reinterpret_cast<float2*>(smem + P.w_tab_bytes - kMaxMels * 8);   // (mean, inv_std), mode 2

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  const int t = lane & 15;
  const int half = lane >> 4;
  unsigned char* const wbase = smem + P.w_tab_bytes + warp * WL::kWarpBytes;
  const TIn* const sm_in = reinterpret_cast<const TIn*>(wbase + WL::off_in);
  float4* const X_pl = reinterpret_cast<float4*>(wbase + WL::off_plane + half * kXPlaneBytes);   // transposition plane
  f2* const my_P = reinterpret_cast<f2*>(X_pl);                                                  // ... and the power pairs
  uint64_t* const bar = reinterpret_cast<uint64_t*>(wbase + WL::off_ctl);
  unsigned char* const slots = wbase + WL::off_ctl + 16;
  int* const wmasks = reinterpret_cast<int*>(wbase + WL::off_aux);
  double* const acc_s = reinterpret_cast<double*>(wbase + WL::off_aux);     // [80] sums
  double* const acc_q = acc_s + kMaxMels;                                    // [80] sums of squares

  const int n_out = (kStdMel != 0) ? 80 : P.n_out;
  const int mode = P.mode;
  constexpr bool kSums = (kStats == 1), kExt = (kStats == 2);

  int taps[kBands], tap_off[kBands + 1];
  tap_off[0] = 0;
#pragma unroll
  for (int b = 0; b < kBands; ++b) {
    taps[b] = kStdMel ? std_taps(kStdMel, b) : P.band_taps[b];
    tap_off[b + 1] = tap_off[b] + taps[b];
  }

  // ---- prologue: tables by one TMA copy, per-warp mbarriers, accumulators at rest ---------------------------------
  if (tid == 0) {
    mbar_init(tab_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(tab_bar, static_cast<uint32_t>(P.const_bytes));
    tma_bulk_g2s_plain(tab, P.const_blob, static_cast<uint32_t>(P.const_bytes), tab_bar);
  }
  if (lane == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (kSums)
    for (int e = lane; e < 2 * kMaxMels; e += 32) acc_s[e] = 0.0;
  if (mode == 2 && tid < n_out) {
    const double n = P.stats_in[2 * n_out];
    const double mean = P.stats_in[tid] / n;
    double var = (P.stats_in[n_out + tid] - P.stats_in[tid] * mean) / (n - 1.0);
    var = var > 0.0 ? var : 0.0;
    sm_norm[tid] = make_float2(static_cast<float>(mean), static_cast<float>(1.0 / (sqrt(var) + 1e-9)));
  }
  __syncthreads();

  // ---- this warp's schedule: its static run of spans [w_first[gw], w_first[gw + 1]), then claims from the pool ----------
  const int gw = blockIdx.x * kWWarps + warp;
  int first_idx = P.n_wspans;                // the span this warp starts with
  int nxt_idx = P.n_wspans;                  // the span after the current one (warp-uniform)
  int pend = P.n_wspans;                     // lane 0: the span after that, fixed early
  int my_end = 0;                            // lane 0: end of the static run
  auto advance = [&](int i) {                // lane 0: the span that follows span i in this warp's schedule
    return (i + 1 < my_end) ? i + 1 : P.n_wstatic + atomicAdd(&P.sched[0], 1);
  };
  if (lane == 0) {
    const int b0 = __ldg(P.w_first + gw);
    my_end = __ldg(P.w_first + gw + 1);
    first_idx = (b0 < my_end) ? b0 : P.n_wstatic + atomicAdd(&P.sched[0], 1);
    if (first_idx < P.n_wspans) {
      nxt_idx = advance(first_idx);
      if (nxt_idx < P.n_wspans) pend = advance(nxt_idx);
    }
  }
  first_idx = __shfl_sync(0xffffffffu, first_idx, 0);
  nxt_idx = __shfl_sync(0xffffffffu, nxt_idx, 0);
  bool have_cur = first_idx < P.n_wspans;
  int cur = 0;                               // which slot holds the current span

  uint32_t phase = 0u;
  const int partner = (lane & 16) | ((16 - t) & 15);
  const int up_lane = (lane & 16) | ((t - 1) & 15);

  auto slot_of = [&](int which) { return reinterpret_cast<const int4*>(slots + 32 * which); };
  // descriptor -> registers (uniform shared-memory loads; the values are only kept as long as they are used)
  auto read_span = [&](int which) {
    const int4 a = slot_of(which)[0], b = slot_of(which)[1];
    WSpanRegs s;
    s.wav_off = (static_cast<long long>(a.y) << 32) | static_cast<unsigned>(a.x);
    s.out_row = (static_cast<long long>(a.w) << 32) | static_cast<unsigned>(a.z);
    s.nframes = b.x; s.utt = b.y; s.t0 = b.z; s.aux = b.w;
    return s;
  };
  // the quad's samples: one TMA bulk copy into the warp's buffer, completion on the warp's mbarrier (lane 0 only)
  auto stage_quad = [&](long long wav_off, int nf) {
    const uint32_t bytes = static_cast<uint32_t>(kFrameShift * nf + (kFrameLen - kFrameShift)) * static_cast<uint32_t>(sizeof(TIn));
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(bar, bytes);
    tma_bulk_g2s(const_cast<TIn*>(sm_in), reinterpret_cast<const TIn*>(P.wav) + wav_off, bytes, bar, l2_evict_first_policy());
  };
  // CENTER framing (kStdMel == 2, the reference's torch.stft branch): quads that touch the constant padding or the
  // reflection at either end of the utterance (spans the host marks aux = 0: the first quad and the last one or two) are
  // staged element by element by the whole warp -- index u of the padded signal p (length N + 2 pad), mirrored once at
  // either end like torch.stft(center=True, pad_mode="reflect"), zeros inside the padding; a plain arrival completes the
  // mbarrier phase.  Interior quads take the TMA copy like the Kaldi framing.   ref: lid/audio_processor.py:91-103
  auto stage_any = [&](const WSpanRegs& sp, int qi) {
    const int nf = min(kQuadFrames, sp.nframes - qi * kQuadFrames);
    if (sp.aux != 0) {
      if (lane == 0) stage_quad(sp.wav_off + static_cast<long long>(qi) * (kQuadFrames * kFrameShift), nf);
    } else {
      const int nsamp = kFrameShift * nf + (kFrameLen - kFrameShift);
      const long long N = P.utt_lengths[sp.utt];
      const TIn* x = reinterpret_cast<const TIn*>(P.wav) + P.utt_offsets[sp.utt];
      const long long Lp = N + 2 * P.pad;
      const long long u0 = static_cast<long long>(kFrameShift) * (sp.t0 + qi * kQuadFrames) - (kFrameLen / 2);
      TIn* dst = const_cast<TIn*>(sm_in);
      for (int i = lane; i < nsamp; i += 32) {
        long long u = u0 + i;
        u = u < 0 ? -u : (u >= Lp ? 2 * (Lp - 1) - u : u);
        const long long r = u - P.pad;
        dst[i] = (r >= 0 && r < N) ? x[r] : static_cast<TIn>(0);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar);
    }
  };
  auto fetch_span = [&](int idx, int which) {    // lane 0: descriptor idx -> slot `which`, asynchronously
    const int4* g = reinterpret_cast<const int4*>(P.wspans + idx);
    cp_async16(const_cast<int4*>(slot_of(which)), g);
    cp_async16(const_cast<int4*>(slot_of(which)) + 1, g + 1);
  };

  mbar_wait(tab_bar, 0u);

  if (have_cur) {
    if (lane == 0) {
      fetch_span(first_idx, 0);
      cp_async_commit();
      cp_async_wait<0>();
    }
    __syncwarp();
    const WSpanRegs s0 = read_span(0);
    if (kStdMel == 2) {
      if (s0.nframes > 0) stage_any(s0, 0);
    } else if (lane == 0 && s0.nframes > 0) stage_quad(s0.wav_off, min(kQuadFrames, s0.nframes));
  }

  int frames_acc = 0;                  // mode 3: frames of the spans this warp has processed
  float ex_max = -INFINITY, ex_min = INFINITY;      // kExt: extrema of held_utt's features seen by this lane
  int held_utt = -1;                   // mode 1: whose sums the accumulators hold

  while (have_cur) {
    // the next span's descriptor travels into the other slot while this span runs
    if (lane == 0) {
      if (nxt_idx < P.n_wspans) fetch_span(nxt_idx, cur ^ 1);
      cp_async_commit();
    }
    const int sp_nframes = read_span(cur).nframes;

    if (__builtin_expect(sp_nframes == 0, 0)) {
      // zero-fill span: pad_sequence's zeros (ref: lid/raw_datasets.py:347-350)
      const WSpanRegs sp = read_span(cur);
      const int total = P.ws_blocked ? 0 : sp.aux * n_out;
      for (int i = lane; i < total; i += 32) {
        const int r = i / n_out;
        P.out[(sp.out_row + r) * P.out_ld + (i - r * n_out)] = 0.f;
      }
      if (kStdMel == 2) {
        if (nxt_idx < P.n_wspans) {
          if (lane == 0) cp_async_wait<0>();
          __syncwarp();
          const WSpanRegs nx = read_span(cur ^ 1);
          if (nx.nframes > 0) stage_any(nx, 0);
        }
      } else if (lane == 0 && nxt_idx < P.n_wspans) {
        cp_async_wait<0>();
        const WSpanRegs nx = read_span(cur ^ 1);
        if (nx.nframes > 0) stage_quad(nx.wav_off, min(kQuadFrames, nx.nframes));
      }
    } else {
      // centred fp32 partial sums of this lane's dims over the last few quads: S = sum(x - c), Q = sum((x - c)^2), c = the
      // first value of the period -- the squares are O(variance), not O(mean^2), so sum(x^2) - sum(x)^2 / n does not cancel
      // the digits an fp32 partial sum has
      float S[kBands], Q[kBands], C[kBands];
    #pragma unroll
      for (int b = 0; b < kBands; ++b) S[b] = Q[b] = C[b] = 0.f;
      int quads_since_fold = 0;
      int cnt = 0;                         // frames this lane has added since the last fold
      // fp32 partials -> lane-owned fp64 accumulators (lanes 0..15 own dims t + 16 b)
      auto fold = [&]() {
        const double n = static_cast<double>(cnt);
    #pragma unroll
        for (int b = 0; b < kBands; ++b) {
          // un-centre in fp64: sum(x) = S + n c,  sum(x^2) = Q + 2 c S + n c^2
          const double c = static_cast<double>(C[b]), sc = static_cast<double>(S[b]);
          double s = fma(n, c, sc);
          double q = fma(n * c, c, fma(2.0 * c, sc, static_cast<double>(Q[b])));
          s += __shfl_xor_sync(0xffffffffu, s, 16);
          q += __shfl_xor_sync(0xffffffffu, q, 16);
          if (half == 0 && t + 16 * b < n_out) {
            acc_s[t + 16 * b] += s;
            acc_q[t + 16 * b] += q;
          }
          S[b] = Q[b] = 0.f;
        }
        quads_since_fold = 0;
        cnt = 0;
      };
      // ---- per-span set-up: the utterance's mask table (modes that mask in the epilogue) --------------------------
      unsigned dim_masked = 0u;
      const int n_masks = (kStats == 0 && (mode == 0 || mode == 2)) ? P.n_masks : 0;
      if (kStats == 0 && n_masks > 0) {
        const int utt = read_span(cur).utt;
        __syncwarp();
        if (lane < n_masks * 4) wmasks[lane] = __ldg(P.masks + static_cast<long long>(utt) * n_masks * 4 + lane);
        __syncwarp();
        for (int q = 0; q < n_masks; ++q) {
          const int f0 = wmasks[4 * q + 2], f1 = wmasks[4 * q + 3];
    #pragma unroll
          for (int b = 0; b < kBands; ++b) dim_masked |= (t + 16 * b >= f0 && t + 16 * b < f1) ? (1u << b) : 0u;
        }
      }
      const int n_quads = (sp_nframes + kQuadFrames - 1) / kQuadFrames;
      // the statistics-free instantiations have the registers the sums would take: the lane's 8 split twiddles stay
      // resident for the span (16 wavefronts per quad less on the shared-memory pipe)
      constexpr bool kTw2Regs = (kStats != 1);
      float2 tw2r[8];
      if constexpr (kTw2Regs) {
    #pragma unroll
        for (int i = 0; i < 8; ++i) tw2r[i] = sm_tw2[i * 16 + t];
      }

      for (int qi = 0; qi < n_quads; ++qi) {
        const int nf = min(kQuadFrames, sp_nframes - qi * kQuadFrames);     // live frames of this quad
        const int flA = half * 2;                                            // frame A inside the quad; B = A + 1
        const bool actA = flA < nf, actB = flA + 1 < nf;
        mbar_wait(bar, phase);
        phase ^= 1u;

        f2 R[16], I[16];
        f2 val[kBands];
        {
          // ---- load (frame B = frame A shifted by 5 loads), DC removal, pre-emphasis, window ----------------------
          const TIn* fr = sm_in + kFrameShift * (actA ? flA : 0);
          float2 x[18];
    #pragma unroll
          for (int j = 0; j < 18; ++j) {
            const int n = t + 16 * j;
            x[j] = (j < 17 || t < 8) ? InTraits<TIn>::ld2(fr + 2 * n, P.in_scale) : make_float2(0.f, 0.f);
          }
          __syncwarp();     // every lane holds its samples: the buffer is free for the next quad
          if (kStdMel == 2) {
            if (qi + 1 < n_quads) {
              stage_any(read_span(cur), qi + 1);
            } else if (nxt_idx < P.n_wspans) {
              if (lane == 0) cp_async_wait<0>();
              __syncwarp();
              const WSpanRegs nx = read_span(cur ^ 1);
              if (nx.nframes > 0) stage_any(nx, 0);
            }
          } else if (lane == 0) {
            if (qi + 1 < n_quads) {
              stage_quad(read_span(cur).wav_off + static_cast<long long>(qi + 1) * (kQuadFrames * kFrameShift),
                         min(kQuadFrames, sp_nframes - (qi + 1) * kQuadFrames));
            } else if (nxt_idx < P.n_wspans) {
              cp_async_wait<0>();
              const WSpanRegs nx = read_span(cur ^ 1);
              if (nx.nframes > 0) stage_quad(nx.wav_off, min(kQuadFrames, nx.nframes));
            }
          }

          float mA = 0.f, mB = 0.f;
          if (kStdMel == 0 && P.remove_dc) {
            f2 sA = make_float2(0.f, 0.f), sB = make_float2(0.f, 0.f);
    #pragma unroll
            for (int j = 0; j < 13; ++j) {
              if (j < 12 || t < 8) {
                sA = add2(sA, x[j]);
                sB = add2(sB, x[j + 5]);
              }
            }
            f2 sum = make_float2(sA.x + sA.y, sB.x + sB.y);
    #pragma unroll
            for (int o = 8; o >= 1; o >>= 1) {
              sum.x += __shfl_xor_sync(0xffffffffu, sum.x, o);
              sum.y += __shfl_xor_sync(0xffffffffu, sum.y, o);
            }
            mA = __fdiv_rn(sum.x, static_cast<float>(kFrameLen));
            mB = __fdiv_rn(sum.y, static_cast<float>(kFrameLen));
          }
          const float c = P.preemph;
          if (kStdMel == 2) {
            // the reference's torch.stft call: window only; the (A, B) pairs are formed by the scalar multiplies themselves
    #pragma unroll
            for (int j = 0; j < 13; ++j) {
              const float2 w = *reinterpret_cast<const float2*>(sm_window + 2 * (t + 16 * j));
              R[j] = make_float2(__fmul_rn(x[j].x, w.x), __fmul_rn(x[j + 5].x, w.x));
              I[j] = make_float2(__fmul_rn(x[j].y, w.y), __fmul_rn(x[j + 5].y, w.y));
            }
          } else if (kStdMel == 1) {
            // The reference's call (DC removal, then pre-emphasis with coefficient 1.0, replicate-left): every output is
            // (x[n] - m) - (x[n-1] - m), and y[0] = (x[0] - m) - (x[0] - m) = 0.  The frame mean m only enters through the
            // rounding of the two inner differences; x[n] - x[n-1] rounded ONCE is the same value with less round-off (the
            // two differ by < 1 ulp of |x|, which is what the reference itself is off by), and the 400-term mean reduction
            // with its 8 shuffles per quad disappears.
            // Frame B is frame A five loads on: element j of B needs the same "previous sample" as element j + 5 of A, so 18
            // shuffles can serve both frames (13 + 13 otherwise); only B's first sample (replicate-left) differs.  Same
            // values either way.  The shared form holds 18 floats at once: it pays in the statistics variant (-2 us on the
            // per-utterance CMVN step) and spills in the statistics-free one, hence the choice per instantiation.
            constexpr bool kPreShare = (kStats == 1);
            if constexpr (kPreShare) {
              float q[18];
    #pragma unroll
              for (int j = 0; j < 18; ++j) {
                const float s = (t == 15) ? (j ? x[j - 1].y : 0.f) : x[j].y;
                q[j] = __shfl_sync(0xffffffffu, s, up_lane);              // x[2n - 1], n = t + 16 j
              }
    #pragma unroll
              for (int j = 0; j < 13; ++j) {
                const float2 w = *reinterpret_cast<const float2*>(sm_window + 2 * (t + 16 * j));
                float qA = q[j], qB = q[j + 5];
                if (j == 0 && t == 0) { qA = x[0].x; qB = x[5].x; }
                const f2 se = make_float2(__fsub_rn(x[j].x, qA), __fsub_rn(x[j + 5].x, qB));
                const f2 so = make_float2(__fsub_rn(x[j].y, x[j].x), __fsub_rn(x[j + 5].y, x[j + 5].x));
                R[j] = mul2(se, bc(w.x));
                I[j] = mul2(so, bc(w.y));
              }
            } else {
              float pA = 0.f, pB = 0.f;
    #pragma unroll
              for (int j = 0; j < 13; ++j) {
                const float2 w = *reinterpret_cast<const float2*>(sm_window + 2 * (t + 16 * j));
                const float sA = (t == 15) ? pA : x[j].y, sB = (t == 15) ? pB : x[j + 5].y;
                float qA = __shfl_sync(0xffffffffu, sA, up_lane);       // x[2n - 1]
                float qB = __shfl_sync(0xffffffffu, sB, up_lane);
                if (j == 0 && t == 0) { qA = x[0].x; qB = x[5].x; }
                pA = x[j].y;
                pB = x[j + 5].y;
                const f2 se = make_float2(__fsub_rn(x[j].x, qA), __fsub_rn(x[j + 5].x, qB));
                const f2 so = make_float2(__fsub_rn(x[j].y, x[j].x), __fsub_rn(x[j + 5].y, x[j + 5].x));
                R[j] = mul2(se, bc(w.x));
                I[j] = mul2(so, bc(w.y));
              }
            }
          } else {
            f2 to_prev = make_float2(0.f, 0.f);
    #pragma unroll
            for (int j = 0; j < 13; ++j) {
              const int n = t + 16 * j;
              const float2 w = *reinterpret_cast<const float2*>(sm_window + 2 * n);
              const f2 te = make_float2(__fsub_rn(x[j].x, mA), __fsub_rn(x[j + 5].x, mB));   // x[2n]   - mean
              const f2 to = make_float2(__fsub_rn(x[j].y, mA), __fsub_rn(x[j + 5].y, mB));   // x[2n+1] - mean
              const f2 send = (t == 15) ? to_prev : to;
              f2 tp;
              tp.x = __shfl_sync(0xffffffffu, send.x, up_lane);
              tp.y = __shfl_sync(0xffffffffu, send.y, up_lane);
              if (j == 0 && t == 0) tp = te;
              to_prev = to;
              const f2 se = sub2(te, mul2(tp, bc(c)));
              const f2 so = sub2(to, mul2(te, bc(c)));
              R[j] = mul2(se, bc(w.x));
              I[j] = mul2(so, bc(w.y));
            }
          }
          if (t >= 8) R[12] = I[12] = make_float2(0.f, 0.f);
          R[13] = R[14] = R[15] = I[13] = I[14] = I[15] = make_float2(0.f, 0.f);
        }

        // ---- stage 1: 16-point DFT over j, twiddle W256^(K1*t), ONE transposition through shared memory --------------
        fft16<true>(R, I);
        {
          // (re_A, re_B) and (im_A, im_B) of a point go out as the two halves of its 16-byte element; the twiddle of point
          // p + 2 is requested before point p is multiplied, so that its shared-memory latency hides behind two complex
          // multiplications instead of stalling each one
          float2 wa = sm_tw1[rev4(1) * 16 + t], wb = sm_tw1[rev4(2) * 16 + t];
          X_pl[t] = make_float4(R[0].x, R[0].y, I[0].x, I[0].y);
    #pragma unroll
          for (int p = 1; p < 16; ++p) {
            const int K1 = rev4(p);
            const float2 w = wa;
            wa = wb;
            if (p + 2 < 16) wb = sm_tw1[rev4(p + 2) * 16 + t];
            cmul2(R[p], I[p], w.x, w.y);
            X_pl[K1 * kXRow + t] = make_float4(R[p].x, R[p].y, I[p].x, I[p].y);
          }
        }
        __syncwarp();
    #pragma unroll
        for (int m = 0; m < 16; ++m) {
          const int e = (m & 3) * 4 + (m >> 2);          // 0, 4, 8, 12, 1, ...: the order the first radix-4 layer consumes
          const float4 v = X_pl[t * kXRow + e];
          R[e] = make_float2(v.x, v.y);
          I[e] = make_float2(v.z, v.w);
        }
        // ---- stage 2 ----------------------------------------------------------------------------------------------
        fft16<false>(R, I);
        __syncwarp();   // every lane has read its row: the plane takes the power bins now

        // ---- real-FFT split + power ---------------------------------------------------------------------------------
        if (t == 0) my_P[128] = mul2(fma2(R[2], R[2], mul2(I[2], I[2])), bc(4.f));
    #pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int ps = rev4(15 - i);
          f2 br, bi;
          br.x = __shfl_sync(0xffffffffu, R[ps].x, partner);
          br.y = __shfl_sync(0xffffffffu, R[ps].y, partner);
          bi.x = __shfl_sync(0xffffffffu, I[ps].x, partner);
          bi.y = __shfl_sync(0xffffffffu, I[ps].y, partner);
          if (t == 0) {
            const int own = (i == 0) ? 0 : rev4(16 - i);
            br = R[own];
            bi = I[own];
          }
          const f2 ar = R[rev4(i)], ai = I[rev4(i)];
          const f2 e2r = add2(ar, br), e2i = sub2(ai, bi);
          f2 o2r = add2(ai, bi), o2i = sub2(br, ar);
          const float2 w = kTw2Regs ? tw2r[i] : sm_tw2[i * 16 + t];
          cmul2(o2r, o2i, w.x, w.y);
          const f2 xar = add2(e2r, o2r), xai = add2(e2i, o2i);
          const f2 xbr = sub2(e2r, o2r), xbi = sub2(e2i, o2i);
          const int k = t + 16 * i;
          my_P[k] = fma2(xar, xar, mul2(xai, xai));
          my_P[256 - k] = fma2(xbr, xbr, mul2(xbi, xbi));
        }
        __syncwarp();

        // ---- sparse triangular mel (segment form) + log ---------------------------------------------------------------
        {
          f2 carry15 = make_float2(0.f, 0.f);
          const int src = (lane & 16) | ((t - 1) & 15);
    #pragma unroll
          for (int b = 0; b < kBands; ++b) {
            f2 own = make_float2(0.f, 0.f), nxt = make_float2(0.f, 0.f);
            const f2* pp = my_P + sm_k0[t + 16 * b];
            const float2* wp = reinterpret_cast<const float2*>(sm_melw) + tap_off[b] * 16 + t;
            if (kStdMel) {
    #pragma unroll
              for (int i = 0; i < std_taps(kStdMel, b); ++i) {
                const f2 p = pp[i];
                const float2 w = wp[i * 16];
                own = fma2(p, bc(w.x), own);
                nxt = fma2(p, bc(w.y), nxt);
              }
            } else {
    #pragma unroll 2
              for (int i = 0; i < taps[b]; ++i) {
                const f2 p = pp[i];
                const float2 w = wp[i * 16];
                own = fma2(p, bc(w.x), own);
                nxt = fma2(p, bc(w.y), nxt);
              }
            }
            f2 got;
            got.x = __shfl_sync(0xffffffffu, nxt.x, src);
            got.y = __shfl_sync(0xffffffffu, nxt.y, src);
            const f2 acc = add2(own, t == 0 ? carry15 : got);
            carry15 = got;
            // variant 1 is the reference's call: log(max(x, FLT_EPSILON)) -- floor, its log and ln 2 are immediates
            const float lfloor = (kStdMel == 1) ? 1.1920928955078125e-07f : P.log_floor;
            const float lof = (kStdMel == 1) ? -15.9423847198486328125f : P.log_of_floor;
            const float lsc = (kStdMel == 1) ? 0.693147180559945309f : P.log_scale;
            val[b] = make_float2(acc.x <= lfloor ? lof : log2_scaled(acc.x, lsc), acc.y <= lfloor ? lof : log2_scaled(acc.y, lsc));
          }
        }
        __syncwarp();   // the power bins have been read: the plane is free for the next quad's transposition

        // ---- epilogue: global CMVN, SpecAugment zero-fill, store ------------------------------------------------------
        {
          const WSpanRegs sp = read_span(cur);
          const int tfA = sp.t0 + qi * kQuadFrames + flA;      // frame index inside the utterance
          const long long row = sp.out_row + qi * kQuadFrames + flA;
          if (P.ws_blocked) {
            // tile-blocked log-mel workspace of the two-kernel MFCC path (see FbankParams::ws_blocked)
            const long long tile_idx = P.utt_first_tile[sp.utt] + tfA / kTileFrames;
            const int fl = tfA % kTileFrames;                   // even: A and B share the tile
            float* o = P.out + tile_idx * (kTileFrames * n_out) + (t >> 2) * 64 + (t & 3) + fl * 4;
    #pragma unroll
            for (int b = 0; b < kBands; ++b) {
              if (t + 16 * b < n_out) {
                if (actA) o[256 * b] = val[b].x;
                if (actB) o[256 * b + 4] = val[b].y;
              }
            }
          } else if (mode != 2 && n_masks == 0 && nf == kQuadFrames) {
            float* orow = P.out + row * P.out_ld + t;
    #pragma unroll
            for (int b = 0; b < kBands; ++b) {
              if (t + 16 * b < n_out) {
                orow[16 * b] = val[b].x;
                orow[P.out_ld + 16 * b] = val[b].y;
              }
            }
          } else {
            bool rowA = false, rowB = false;
            for (int q = 0; q < n_masks; ++q) {
              const int m0 = wmasks[4 * q], m1 = wmasks[4 * q + 1];
              rowA |= (tfA >= m0 && tfA < m1);
              rowB |= (tfA + 1 >= m0 && tfA + 1 < m1);
            }
            float* orow = P.out + row * P.out_ld + t;
    #pragma unroll
            for (int b = 0; b < kBands; ++b) {
              const int d = t + 16 * b;
              if (d < n_out) {
                f2 xv = val[b];
                if (mode == 2) {
                  const float2 nm = sm_norm[d];
                  xv = mul2(sub2(xv, bc(nm.x)), bc(nm.y));
                }
                const bool dz = (dim_masked >> b) & 1u;
                if (actA) orow[16 * b] = (dz || rowA) ? 0.f : xv.x;
                if (actB) orow[P.out_ld + 16 * b] = (dz || rowB) ? 0.f : xv.y;
              }
            }
          }
        }

        // ---- AmplitudeToDB(top_db): running extrema of this lane's live features (ta: functional/functional.py:391-403) ------
        if (kExt) {
    #pragma unroll
          for (int b = 0; b < kBands; ++b)
            if (t + 16 * b < n_out) {
              if (actA) { ex_max = fmaxf(ex_max, val[b].x); ex_min = fminf(ex_min, val[b].x); }
              if (actB) { ex_max = fmaxf(ex_max, val[b].y); ex_min = fminf(ex_min, val[b].y); }
            }
        }
        // ---- statistics: centred fp32 partial sums in registers, folded into fp64 every kFoldQuads quads -------------
        if (kSums) {
          if (quads_since_fold == 0) {     // (a dead pair holds frame 0 of its quad: as good a centre as any)
    #pragma unroll
            for (int b = 0; b < kBands; ++b) C[b] = val[b].x;
          }
          if (nf == kQuadFrames) {
    #pragma unroll
            for (int b = 0; b < kBands; ++b) {
              const float dx = val[b].x - C[b], dy = val[b].y - C[b];
              S[b] += dx + dy;
              Q[b] = fmaf(dx, dx, fmaf(dy, dy, Q[b]));
            }
            cnt += 2;
          } else {
    #pragma unroll
            for (int b = 0; b < kBands; ++b) {
              const float dx = val[b].x - C[b], dy = val[b].y - C[b];
              if (actA) { S[b] += dx; Q[b] = fmaf(dx, dx, Q[b]); }
              if (actB) { S[b] += dy; Q[b] = fmaf(dy, dy, Q[b]); }
            }
            cnt += (actA ? 1 : 0) + (actB ? 1 : 0);
          }
          if (++quads_since_fold == kFoldQuads) fold();
        }
      }   // quads of the span
      if (kExt) held_utt = read_span(cur).utt;
      if (kSums) {
        // every span's contribution is folded before the next one starts: what a span adds to the sums is then a function
        // of the span alone, not of which warp happened to claim it after what (bit-reproducible statistics up to the
        // order of the fp64 additions)
        if (quads_since_fold) fold();
        frames_acc += sp_nframes;
        held_utt = read_span(cur).utt;
      }
    }

    // ---- end of span: the next descriptor (already in the other slot), the claim after it, statistics hand-over -------
    const bool have_next = nxt_idx < P.n_wspans;
    if (have_next) {
      if (lane == 0) cp_async_wait<0>();
      __syncwarp();
    }
    if (kExt && held_utt >= 0) {
      bool hand_over = !have_next;
      if (have_next) {
        const WSpanRegs nx = read_span(cur ^ 1);
        hand_over = (nx.nframes == 0) || (nx.utt != held_utt);
      }
      if (hand_over) {
    #pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
          ex_max = fmaxf(ex_max, __shfl_xor_sync(0xffffffffu, ex_max, o));
          ex_min = fminf(ex_min, __shfl_xor_sync(0xffffffffu, ex_min, o));
        }
        if (lane == 0) {
          atomicMax(P.utt_max + (P.parity & 1) * P.b_cap + held_utt, f2ord(ex_max));
          atomicMin(P.utt_min + (P.parity & 1) * P.b_cap + held_utt, f2ord(ex_min));
        }
        ex_max = -INFINITY;
        ex_min = INFINITY;
        held_utt = -1;
      }
    }
    if (kSums && mode == 1 && held_utt >= 0) {
      bool hand_over = !have_next;
      if (have_next) {
        const WSpanRegs nx = read_span(cur ^ 1);
        hand_over = (nx.nframes == 0) || (nx.utt != held_utt);
      }
      if (hand_over) {
        __syncwarp();
        double* g = P.utt_stats + (static_cast<long long>(P.parity & 1) * P.b_cap + held_utt) * 2 * n_out;
        for (int e = lane; e < n_out; e += 32) {
          const double a = acc_s[e], b2 = acc_q[e];
          acc_s[e] = 0.0; acc_q[e] = 0.0;
          if (a != 0.0) atomicAdd(g + e, a);
          if (b2 != 0.0) atomicAdd(g + n_out + e, b2);
        }
        held_utt = -1;
      }
    }
    __syncwarp();      // every lane is done with the current slot before lane 0 lets a descriptor overwrite it
    have_cur = have_next;
    cur ^= 1;
    if (lane == 0) {
      nxt_idx = pend;
      if (nxt_idx < P.n_wspans) pend = advance(nxt_idx);
    }
    nxt_idx = __shfl_sync(0xffffffffu, nxt_idx, 0);
  }

  // ---- out of work: global sums leave the CTA once; the last CTA puts the claim counter back to rest ----------------
  if (kSums && mode == 3) {
    __syncthreads();
    for (int e = tid; e < 2 * kMaxMels; e += kWThreads) {
      const int which = e / kMaxMels, d = e - which * kMaxMels;
      double a = 0.0;
#pragma unroll
      for (int w = 0; w < kWWarps; ++w)
        a += reinterpret_cast<const double*>(smem + P.w_tab_bytes + w * WL::kWarpBytes + WL::off_aux)[e];
      if (d < n_out && a != 0.0) atomicAdd(&P.stats_out[which * n_out + d], a);
    }
    if (lane == 0 && frames_acc != 0) atomicAdd(&P.stats_out[2 * n_out], static_cast<double>(frames_acc));
  }
  __syncthreads();
  if (tid == 0) {
    if (atomicAdd(&P.sched[1], 1) == static_cast<int>(gridDim.x) - 1) {
      P.sched[0] = 0;
      P.sched[1] = 0;
    }
  }
}

}  // namespace lidfe
