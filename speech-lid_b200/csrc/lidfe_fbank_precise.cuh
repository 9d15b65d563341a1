// lidfe_fbank_precise.cuh -- the "precise" arithmetic mode of the Kaldi fbank / MFCC path (lidfe_set_precision(h, 1)).
//
// Why it exists (DESIGN.md section 2): SURVEY.md 8(c)'s acceptance metric (iv) -- per mel bin, |gpu - truth64| <= 1.5 x
// |oracle32 - truth64| over all frames -- is a race between two fp32 FFTs; measured on the CPU alone, scipy's pocketfft
// loses it against torch's FFT on 5.7 % of the (utterance, bin) pairs, and the fast kernel's 16 x 16 FFT on 6.8 %.  No
// fp32 FFT that is not the oracle's own wins it everywhere.  This kernel takes the other way out: it evaluates the
// reference's formula (ref: lid/audio_processor.py:41-69 -> ta: compliance/kaldi.py:183-217, 514-645) in FLOAT64 from the
// samples to the logarithm (and through the DCT for MFCC) with the reference's own fp32 tables (window, mel bank, DCT,
// lifter) and rounds ONCE, at the store.  Its distance to the fp64 truth is half an ulp of the feature, whatever the
// oracle's host FFT does, so (iv) holds by construction; what remains of metric (ii) is the reference's own fp32 error.
//
// Same decomposition as the fast kernels -- the 512-point real FFT as a 256-point complex FFT of z[n] = x[2n] + i x[2n+1],
// 16 x 16 with an in-register radix-4 x 4 DFT per lane, one transposition through shared memory, real-FFT split by
// shuffles between lane t and lane 16 - t -- but one frame per half-warp in doubles instead of a frame pair in packed
// floats, the mel bank in the fast kernels' segment form with fp64 accumulation, libdevice's log.  B200's FP64 pipe runs DFMA at half
// the FFMA rate (tools/ubench.cu: 62.5 against 120 lane-ops/clk/SM), so this is a 3-4 x slower kernel, not a 30 x one (measured: 340 us against 100 us per 256 x 8 s).
// Scope: KALDI framing (the reference's Kaldi call and its relatives) and CENTER framing (its default branch: window-only
// framing, HTK mel, dB, per-utterance extrema for AmplitudeToDB's top_db clamp), float32 / int16 input, fbank or MFCC
// output, every CMVN mode (statistics / extrema are taken here, the normalisation / clamp / masks run in
// cmvn_apply_kernel as for the fast path).
#pragma once
#include "lidfe_kernels.cuh"

namespace lidfe {

struct PreciseParams {
  const void* wav;
  float* out;
  long long out_ld;
  const Span* spans;
  int n_spans;
  const float* window;      // [400]                      the handle's fp32 window (blob offset 0)
  const int* mel_k0;        // [80]                       the handle's segment-form mel plan (build_mel_plan, lidfe_abi.cu):
  const float* mel_w;       // [total_taps][16][2]        per lane its first power bin and per step the (own, next) weights,
  int band_taps[kBands];    //                            x 0.25 (the power bins are left scaled by 4) -- exact in any precision
  int total_taps;
  const float* dct;         // [n_mels][n_ceps] or NULL
  const float* lifter;      // [n_ceps]
  int n_mels, n_ceps, n_out;
  float preemph, in_scale, log_floor, log_of_floor;
  int remove_dc;
  double log_mul;           // 1 (natural log) or 10 / ln 10 (dB)
  int center, pad;          // LIDFE_FRAMING_CENTER: frame f covers p[160 f - 200, 160 f + 200) of the constant-padded, reflect-extended signal
  const long long* utt_offsets;   // [B] (CENTER framing)
  const long long* utt_lengths;   // [B]
  unsigned* utt_max;        // this launch's half, [B_cap]: order-preserving encoding of the utterance's max / min feature
  unsigned* utt_min;        //   (mode 4, AmplitudeToDB's top_db clamp runs in cmvn_apply_kernel)
  int mode;                 // LIDFE_CMVN_*: 1 -> sums into utt_stats, 3 -> sums into stats_out, 4 -> extrema
  double* utt_stats;        // this launch's half: [B_cap][2][n_out]
  double* stats_out;        // [2 * n_out + 1]
};

constexpr int kPThreads = 128;
constexpr int kPCtasPerSm = 4;
constexpr int kPHalfWarps = kPThreads / 16;
constexpr int kPRow = 17;                               // double2 elements per transposition row (conflict-free both ways)
constexpr int kPPlane = 16 * kPRow;                     // double2 elements per half-warp plane (4352 bytes)
constexpr int kPLogmelOff = 264;                        // doubles: the 80 log-mels of the MFCC epilogue sit behind the 257 power bins

__device__ __forceinline__ void radix4d(double& r0, double& i0, double& r1, double& i1, double& r2, double& i2, double& r3, double& i3) {
  const double t0r = r0 + r2, t0i = i0 + i2, t1r = r0 - r2, t1i = i0 - i2;
  const double t2r = r1 + r3, t2i = i1 + i3, t3r = r1 - r3, t3i = i1 - i3;
  r0 = t0r + t2r; i0 = t0i + t2i;
  r2 = t0r - t2r; i2 = t0i - t2i;
  r1 = t1r + t3i; i1 = t1i - t3r;
  r3 = t1r - t3i; i3 = t1i + t3r;
}
__device__ __forceinline__ void cmuld(double& R, double& I, double wr, double wi) {
  const double nr = R * wr - I * wi, ni = R * wi + I * wr;
  R = nr;
  I = ni;
}
// forward 16-point DFT, natural order in, position p holds X[rev4(p)] (same structure as fft16 in lidfe_kernels.cuh)
__device__ __forceinline__ void fft16d(double (&R)[16], double (&I)[16]) {
  constexpr double kC1 = 0.92387953251128675613;   // cos(pi/8)
  constexpr double kS1 = 0.38268343236508977173;   // sin(pi/8)
  constexpr double kH = 0.70710678118654752440;    // sqrt(1/2)
#pragma unroll
  for (int q = 0; q < 4; ++q) radix4d(R[q], I[q], R[q + 4], I[q + 4], R[q + 8], I[q + 8], R[q + 12], I[q + 12]);
  // element n2 + 4 k1 *= W16^(n2 k1)
  cmuld(R[5], I[5], kC1, -kS1);      // W^1
  cmuld(R[9], I[9], kH, -kH);        // W^2
  cmuld(R[13], I[13], kS1, -kC1);    // W^3
  cmuld(R[6], I[6], kH, -kH);        // W^2
  cmuld(R[10], I[10], 0.0, -1.0);    // W^4
  cmuld(R[14], I[14], -kH, -kH);     // W^6
  cmuld(R[7], I[7], kS1, -kC1);      // W^3
  cmuld(R[11], I[11], -kH, -kH);     // W^6
  cmuld(R[15], I[15], -kC1, kS1);    // W^9
#pragma unroll
  for (int q = 0; q < 4; ++q) radix4d(R[4 * q], I[4 * q], R[4 * q + 1], I[4 * q + 1], R[4 * q + 2], I[4 * q + 2], R[4 * q + 3], I[4 * q + 3]);
}

template <typename TIn>
__device__ __forceinline__ double ld_sample(const TIn* p, float scale);
template <>
__device__ __forceinline__ double ld_sample<float>(const float* p, float) { return static_cast<double>(__ldg(p)); }
template <>
__device__ __forceinline__ double ld_sample<short>(const short* p, float scale) {
  return static_cast<double>(static_cast<float>(__ldg(p)) * scale);      // the fp32 product torchaudio.load forms (exact for 2^-15)
}

// dynamic shared memory: tw1[16][16] double2 (stage twiddles W256^(K1 t), lane-major: conflict-free) | tw2[128] double2
// (split twiddles W512^k) | window[400] double | mel plan weights [kPMaxTaps][16] float2 | mel first bins [80] int | planes
constexpr int kPMaxTaps = 64;      // steps of the segment plan summed over the five bands (Kaldi-80: 23)
constexpr int kPMelW = kPMaxTaps * 16;
constexpr int kPOffTw2 = 256 * 16;
constexpr int kPOffWin = kPOffTw2 + 128 * 16;
constexpr int kPOffMelW = kPOffWin + 400 * 8;
constexpr int kPOffMelR = kPOffMelW + kPMelW * 8;
constexpr int kPOffPlane = kPOffMelR + kMaxMels * 4 + 64;
constexpr int kPSmemBytes = kPOffPlane + kPHalfWarps * kPPlane * 16;

template <typename TIn, bool kCenter>
__global__ void __launch_bounds__(kPThreads, kPCtasPerSm) fbank_precise_kernel(const PreciseParams P) {
  extern __shared__ __align__(16) unsigned char psmem[];
  double2* const sm_tw1 = reinterpret_cast<double2*>(psmem);                       // [K1][t]: W256^(K1 t) = (cos, -sin)(2 pi K1 t / 256)
  double2* const sm_tw2 = reinterpret_cast<double2*>(psmem + kPOffTw2);            // W512^k = (cos, -sin)(2 pi k / 512), k = 0..127
  double* const sm_win = reinterpret_cast<double*>(psmem + kPOffWin);
  float2* const sm_melw = reinterpret_cast<float2*>(psmem + kPOffMelW);            // [step][lane] (own, next) weights
  int* const sm_k0 = reinterpret_cast<int*>(psmem + kPOffMelR);                    // [80] first power bin of lane t, band b
  double2* const sm_plane = reinterpret_cast<double2*>(psmem + kPOffPlane);

  const int tid = threadIdx.x, lane = tid & 31, t = lane & 15;
  const int hw = tid >> 4;
  double2* const X_pl = sm_plane + hw * kPPlane;
  double* const Pw = reinterpret_cast<double*>(X_pl);
  double* const LM = Pw + kPLogmelOff;
  const int partner = (lane & 16) | ((16 - t) & 15);
  const int up_lane = (lane & 16) | ((t - 1) & 15);
  const bool stats = (P.mode == 1 || P.mode == 3);

  for (int k = tid; k < 256; k += kPThreads) {
    double s, c;
    sincospi(static_cast<double>((k >> 4) * (k & 15)) / 128.0, &s, &c);
    sm_tw1[k] = make_double2(c, -s);
    if (k < 128) {
      sincospi(static_cast<double>(k) / 256.0, &s, &c);
      sm_tw2[k] = make_double2(c, -s);
    }
  }
  for (int k = tid; k < kFrameLen; k += kPThreads) sm_win[k] = static_cast<double>(__ldg(P.window + k));
  for (int e = tid; e < P.total_taps * 16; e += kPThreads) sm_melw[e] = __ldg(reinterpret_cast<const float2*>(P.mel_w) + e);
  for (int e = tid; e < kMaxMels; e += kPThreads) sm_k0[e] = __ldg(P.mel_k0 + e);
  int tap_off[kBands + 1];
  tap_off[0] = 0;
#pragma unroll
  for (int b = 0; b < kBands; ++b) tap_off[b + 1] = tap_off[b] + P.band_taps[b];
  const int src = (lane & 16) | ((t - 1) & 15);
  __syncthreads();

  const double cpre = static_cast<double>(P.preemph);
  const TIn* const wav = reinterpret_cast<const TIn*>(P.wav);

  // work unit = one of the kMaxSpanTiles 16-frame tiles of a span (a span is <= 128 frames of one utterance), dealt out
  // round-robin: ~20 units per CTA on cfg2, so the last round costs a few per cent (whole spans: 3 per CTA, +30 %)
  const int n_units = P.n_spans * kMaxSpanTiles;
  for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
    const int ch = u / P.n_spans, si = u - ch * P.n_spans;     // tile-major: the live units (spans may hold fewer than 8 tiles) stay contiguous in u
    const Span sp = P.spans[si];
    if (sp.nframes == 0) {        // pad_sequence's zero rows (ref: lid/raw_datasets.py:347-350), an eighth of them per unit
      const int r0 = static_cast<int>(static_cast<long long>(sp.aux) * ch / kMaxSpanTiles);
      const int r1 = static_cast<int>(static_cast<long long>(sp.aux) * (ch + 1) / kMaxSpanTiles);
      for (int r = r0; r < r1; ++r)
        for (int d = tid; d < P.n_out; d += kPThreads) P.out[(sp.out_row + r) * P.out_ld + d] = 0.f;
      continue;
    }
    const int fbeg = ch * kTileFrames;
    if (fbeg >= sp.nframes) continue;
    const int fend = min(sp.nframes, fbeg + kTileFrames);
    double ssum[kBands], qsum[kBands];      // this lane's share of the unit's sums (dims t + 16 b, frames of its half-warp)
    float ex_max = -INFINITY, ex_min = INFINITY;
#pragma unroll
    for (int b = 0; b < kBands; ++b) ssum[b] = qsum[b] = 0.0;
    for (int f0 = fbeg; f0 < fend; f0 += kPHalfWarps) {
      const bool active = f0 + hw < fend;
      const int f = active ? f0 + hw : fend - 1;
      const TIn* const x = wav + sp.wav_off + static_cast<long long>(kFrameShift) * f;
      // CENTER framing (the reference's torch.stft branch, ref: lid/audio_processor.py:91-103): sample i of frame tf is
      // p[160 tf - 200 + i], p = the utterance with `pad` zeros on either side, mirrored once at either end
      const long long cN = kCenter ? __ldg(P.utt_lengths + sp.utt) : 0;
      const TIn* const cx = kCenter ? wav + __ldg(P.utt_offsets + sp.utt) : wav;
      const long long cLp = cN + 2 * P.pad;
      const long long cu0 = static_cast<long long>(kFrameShift) * (sp.t0 + f) - (kFrameLen / 2);
      // (interior frames -- all but the first two and the last two or three of an utterance -- touch neither the padding
      // nor the reflection: plain loads)
      const bool interior = kCenter && (cu0 - P.pad >= 0) && (cu0 - P.pad + kFrameLen <= cN);
      const TIn* const xe = kCenter ? cx + (cu0 - P.pad) : x;
      // ONE branch per frame, so that either path issues its 26 loads back to back (a branch per sample serialised
      // them: 2 x the kernel time)
      double R[16], I[16];
      double a0[13], a1[13], pm[13];
      if (!kCenter || interior) {
#pragma unroll
        for (int j = 0; j < 13; ++j) {
          const int n = t + 16 * j;
          const bool valid = (j < 12 || t < 8);
          a0[j] = valid ? ld_sample<TIn>(xe + 2 * n, P.in_scale) : 0.0;
          a1[j] = valid ? ld_sample<TIn>(xe + 2 * n + 1, P.in_scale) : 0.0;
        }
      } else {
        auto sample = [&](int i) -> double {
          long long u = cu0 + i;
          u = u < 0 ? -u : (u >= cLp ? 2 * (cLp - 1) - u : u);
          const long long r = u - P.pad;
          return (r >= 0 && r < cN) ? ld_sample<TIn>(cx + r, P.in_scale) : 0.0;
        };
#pragma unroll
        for (int j = 0; j < 13; ++j) {
          const int n = t + 16 * j;
          const bool valid = (j < 12 || t < 8);
          a0[j] = valid ? sample(2 * n) : 0.0;
          a1[j] = valid ? sample(2 * n + 1) : 0.0;
        }
      }
#pragma unroll
      for (int j = 0; j < 13; ++j) {      // x[2n - 1] sits in lane t - 1 (lane 15 of the previous j for t = 0); x[-1] := x[0]
        const double send = (t == 15) ? (j ? a1[j - 1] : 0.0) : a1[j];
        pm[j] = __shfl_sync(0xffffffffu, send, up_lane);
        if (j == 0 && t == 0) pm[j] = a0[0];
      }
      double mean = 0.0;
      if (P.remove_dc) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 13; ++j) s += a0[j] + a1[j];
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        mean = s / static_cast<double>(kFrameLen);
      }
#pragma unroll
      for (int j = 0; j < 13; ++j) {
        const int n = t + 16 * j;
        const bool valid = (j < 12 || t < 8);
        const double2 w = valid ? *reinterpret_cast<const double2*>(sm_win + 2 * n) : make_double2(0.0, 0.0);
        const double w0 = w.x, w1 = w.y;
        const double e = a0[j] - mean, o = a1[j] - mean, p = pm[j] - mean;
        R[j] = (e - cpre * p) * w0;
        I[j] = (o - cpre * e) * w1;
      }
      R[13] = R[14] = R[15] = I[13] = I[14] = I[15] = 0.0;

      // ---- 256-point complex FFT as 16 x 16 -------------------------------------------------------------------------
      fft16d(R, I);
      X_pl[t] = make_double2(R[0], I[0]);
#pragma unroll
      for (int p = 1; p < 16; ++p) {
        const int K1 = rev4(p);
        const double2 w = sm_tw1[K1 * 16 + t];
        cmuld(R[p], I[p], w.x, w.y);
        X_pl[K1 * kPRow + t] = make_double2(R[p], I[p]);
      }
      __syncwarp();
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const double2 v = X_pl[t * kPRow + e];
        R[e] = v.x;
        I[e] = v.y;
      }
      fft16d(R, I);       // position p holds Z[t + 16 rev4(p)]
      __syncwarp();       // every lane has read its row: the plane takes the power bins now

      // ---- real-FFT split + |X|^2 -----------------------------------------------------------------------------------
      if (t == 0) Pw[128] = 4.0 * (R[2] * R[2] + I[2] * I[2]);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int ps = rev4(15 - i);
        double br = __shfl_sync(0xffffffffu, R[ps], partner);
        double bi = __shfl_sync(0xffffffffu, I[ps], partner);
        if (t == 0) {
          const int own = (i == 0) ? 0 : rev4(16 - i);
          br = R[own];
          bi = I[own];
        }
        const double ar = R[rev4(i)], ai = I[rev4(i)];
        const double e2r = ar + br, e2i = ai - bi;
        double o2r = ai + bi, o2i = br - ar;
        const int k = t + 16 * i;
        const double2 w = sm_tw2[k];
        cmuld(o2r, o2i, w.x, w.y);
        const double xar = e2r + o2r, xai = e2i + o2i, xbr = e2r - o2r, xbi = e2i - o2i;
        Pw[k] = xar * xar + xai * xai;              // 4 |X[k]|^2: the plan's weights carry the 1/4
        Pw[256 - k] = xbr * xbr + xbi * xbi;
      }
      __syncwarp();

      // ---- mel in segment form (lane t of band b walks the bins between the centres of filters m = t + 16 b and m + 1 once:
      //      the down-slope share of its own filter and the up-slope share of the next one, handed one lane up; the same
      //      conflict-free plan as the fast kernels), log, optional DCT-II + lifter; ONE rounding, at the store -----------
      float val[kBands];
      double carry15 = 0.0;
#pragma unroll
      for (int b = 0; b < kBands; ++b) {
        const int m = t + 16 * b;
        double own = 0.0, nxt = 0.0;
        const double* pp = Pw + sm_k0[m];
        const float2* wp = sm_melw + tap_off[b] * 16 + t;
        for (int i = 0; i < P.band_taps[b]; ++i) {
          const double p = pp[i];
          const float2 w = wp[i * 16];
          own = fma(p, static_cast<double>(w.x), own);
          nxt = fma(p, static_cast<double>(w.y), nxt);
        }
        const double got = __shfl_sync(0xffffffffu, nxt, src);
        const double E = own + (t == 0 ? carry15 : got);
        carry15 = got;
        double v = 0.0;
        val[b] = 0.f;
        if (m < P.n_mels) {
          const bool floored = !(E > static_cast<double>(P.log_floor));
          v = floored ? static_cast<double>(P.log_of_floor) : log(E) * P.log_mul;
          val[b] = floored ? P.log_of_floor : static_cast<float>(v);
          if (P.n_ceps > 0) LM[m] = v;
        }
      }
      if (P.n_ceps > 0) {
        __syncwarp();
#pragma unroll
        for (int b = 0; b < kBands; ++b) {
          const int j = t + 16 * b;
          val[b] = 0.f;
          if (j < P.n_ceps) {
            double c = 0.0;     // (four independent chains were measured: 959 us against 743 us per 512 x 4 s -- register pressure)
            for (int m = 0; m < P.n_mels; ++m) c = fma(LM[m], static_cast<double>(__ldg(P.dct + m * P.n_ceps + j)), c);
            val[b] = static_cast<float>(c * static_cast<double>(__ldg(P.lifter + j)));
          }
        }
      }
      if (active) {
        float* orow = P.out + (sp.out_row + f) * P.out_ld;
#pragma unroll
        for (int b = 0; b < kBands; ++b) {
          const int d = t + 16 * b;
          if (d < P.n_out) {
            orow[d] = val[b];
            const double xv = static_cast<double>(val[b]);
            ssum[b] += xv;
            qsum[b] = fma(xv, xv, qsum[b]);
            ex_max = fmaxf(ex_max, val[b]);
            ex_min = fminf(ex_min, val[b]);
          }
        }
      }
      __syncwarp();       // the power bins / log-mels have been read: the plane is free for the next frame
    }
    if (P.mode == 4) {        // AmplitudeToDB(top_db): the utterance's extrema (ta: functional/functional.py:391-403)
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        ex_max = fmaxf(ex_max, __shfl_xor_sync(0xffffffffu, ex_max, o));
        ex_min = fminf(ex_min, __shfl_xor_sync(0xffffffffu, ex_min, o));
      }
      if (lane == 0) {
        atomicMax(P.utt_max + sp.utt, f2ord(ex_max));
        atomicMin(P.utt_min + sp.utt, f2ord(ex_min));
      }
    }
    if (stats) {
      // the half-warps park their sums in their (now idle) planes; 160 threads-worth of adds, then one atomic per dim
#pragma unroll
      for (int b = 0; b < kBands; ++b) {
        Pw[t + 16 * b] = ssum[b];
        Pw[kMaxMels + t + 16 * b] = qsum[b];
      }
      __syncthreads();
      for (int e = tid; e < 2 * kMaxMels; e += kPThreads) {
        const int which = e / kMaxMels, d = e - which * kMaxMels;
        double a = 0.0;
#pragma unroll
        for (int h = 0; h < kPHalfWarps; ++h) a += reinterpret_cast<const double*>(sm_plane + h * kPPlane)[e];
        if (d < P.n_out && a != 0.0) {
          if (P.mode == 1) atomicAdd(P.utt_stats + (static_cast<long long>(sp.utt) * 2 + which) * P.n_out + d, a);
          else atomicAdd(P.stats_out + which * P.n_out + d, a);
        }
      }
      if (P.mode == 3 && tid == 0) atomicAdd(P.stats_out + 2 * P.n_out, static_cast<double>(fend - fbeg));
      __syncthreads();
    }
  }
}

}  // namespace lidfe
