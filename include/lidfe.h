/*
 * lidfe.h -- C ABI of the B200-native speech-lid front-end (liblidfe.so).
 *
 * Drop-in boundary for ONE path of kouyt5/speech-lid: raw 16 kHz waveform -> kaldi log-mel
 * fbank / MFCC -> SpecAugment masks -> CMVN -> (rows, n_out) features.  Each entry point names
 * the reference interface it replaces ("ref:" = path in the reference tree, "ta:" = path inside the
 * torchaudio package the reference calls; the reference has no native code, its "FFI" is the Python
 * call boundary of lid/audio_processor.py, so the binding a maintainer adds is a ctypes stub --
 * INTEGRATION.md shows it).
 *
 * Conventions
 *   - Plain C types only.  Pointers named *_dev are DEVICE pointers owned by the caller (PyTorch
 *     tensors' data_ptr()); *_host are host pointers.  `stream` is a cudaStream_t passed as void*.
 *   - Return value: 0 = OK; < 0 = contract error (LIDFE_E_*); > 0 = a cudaError_t.  Nothing throws,
 *     nothing calls exit().  lidfe_strerror() maps any return value to text.
 *   - A handle is immutable after lidfe_create(); a plan is immutable after lidfe_plan_create().
 *     All device work is enqueued asynchronously on `stream`.  lidfe_create uploads its tables and returns after they
 *     have landed (one synchronisation, once).  lidfe_plan_create_async fills a pinned staging buffer and enqueues ONE
 *     copy on the caller's stream: plans take their device / pinned memory from a pool owned by the handle, so a new
 *     batch shape every step (ragged training batches) costs no cudaMalloc / cudaFree / device synchronisation once the
 *     pool is warm.  lidfe_plan_create is the same followed by a wait on that copy.
 *   - Ordering contract: a plan's tables are uploaded on the stream handed to lidfe_plan_create_async; use the plan
 *     on that stream (or order other streams after it yourself).  A plan owns device workspace, so it is in flight on
 *     one stream at a time.
 *   - There is no CPU implementation behind this ABI.  Without a CUDA device every compute entry
 *     point returns a cudaError_t.
 */
#ifndef LIDFE_H_
#define LIDFE_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LIDFE_ABI_VERSION 8

/* error codes (negative) */
#define LIDFE_OK 0
#define LIDFE_E_NULL -1        /* required pointer is NULL */
#define LIDFE_E_CONFIG -2      /* unsupported configuration (sample rate, frame geometry, n_mels ...) */
#define LIDFE_E_SHORT -3       /* an utterance is shorter than one frame (ta: compliance/kaldi.py:142 asserts) */
#define LIDFE_E_OFFSETS -4     /* offsets not monotone / overlapping / negative */
#define LIDFE_E_ARG -5         /* bad scalar argument (B <= 0, ld < n_out, unknown mode ...) */
#define LIDFE_E_MELBANK -6     /* mel bank row is empty, non-contiguous beyond limits or too wide */
#define LIDFE_E_NOMEM -7       /* host allocation failed */

/* input sample types */
#define LIDFE_IN_F32 0
#define LIDFE_IN_I16 1         /* int16 PCM, converted in-kernel as (float)s * in_scale */

/* cmvn modes of lidfe_featurize */
#define LIDFE_CMVN_NONE 0          /* ref behaviour: features leave the kernel un-normalised */
#define LIDFE_CMVN_PER_UTT 1       /* per utterance, per output dim: (x - mean_t) / (std_t + 1e-9), unbiased */
#define LIDFE_CMVN_APPLY_GLOBAL 2  /* normalise in the fbank epilogue with caller-supplied global sums */
#define LIDFE_CMVN_ACCUM_GLOBAL 3  /* write raw features, add [sum, sumsq, count] to stats_out_dev */
#define LIDFE_POST_TOPDB 4         /* AmplitudeToDB(top_db): clamp every value of an utterance at (its max - cfg.top_db) */

/* framing */
#define LIDFE_FRAMING_KALDI 0      /* snip_edges=True: frame f = x[160 f, 160 f + 400), 1 + (N-400)/160 frames */
#define LIDFE_FRAMING_CENTER 1     /* torch.stft(center=True, reflect): frame f centred at 160 f over the (constant-
                                      padded) signal, 1 + (N + 2 pad)/160 frames; window centred in the 512-point FFT */
/* log flavours */
#define LIDFE_LOG_NATURAL 0        /* log(max(x, log_floor))           (kaldi fbank) */
#define LIDFE_LOG_DB10 1           /* 10*log10(max(x, log_floor))      (AmplitudeToDB, power) */

typedef struct lidfe_ctx* lidfe_handle;
typedef struct lidfe_plan_s* lidfe_plan;

/*
 * Front-end configuration.  Mirrors the argument set the reference passes to
 * torchaudio.compliance.kaldi.fbank (ref: lid/audio_processor.py:41-69; ta: compliance/kaldi.py:514-541).
 * The same struct configures the reference's default branch, MelSpectrogram + AmplitudeToDB(top_db=80)
 * (ref: lid/audio_processor.py:72-105): framing CENTER, preemph 0, remove_dc 0, periodic Hann window, HTK mel bank,
 * log_kind DB10, log_floor 1e-10, top_db 80 -- the |FFT|^2 of a frame does not depend on where the 400-sample window
 * sits inside the 512-point buffer, so the kernel is shared.
 * Supported geometry this round: sample_rate 16000, frame_len 400, frame_shift 160, fft_len 512,
 * 4 <= n_mels <= 80, n_ceps 0 (fbank) or 1..n_mels (MFCC).  Anything else -> LIDFE_E_CONFIG (the survey
 * asks for a loud error rather than silent mis-framing at other rates).
 */
typedef struct {
  int sample_rate;   /* 16000 */
  int frame_len;     /* 400  = int(sr * 25 ms)                                  */
  int frame_shift;   /* 160  = int(sr * 10 ms)                                  */
  int fft_len;       /* 512  = next power of two (round_to_power_of_two=True)   */
  int n_mels;        /* 80                                                       */
  int n_ceps;        /* 0 -> log-mel fbank; >0 -> MFCC with n_ceps coefficients  */
  float preemph;     /* 1.0 in the reference's call (per frame, replicate-left)  */
  int remove_dc;     /* 1                                                        */
  float log_floor;   /* 1.1920929e-07 (FLT_EPSILON)                              */
  int in_dtype;      /* LIDFE_IN_F32 | LIDFE_IN_I16                              */
  float in_scale;    /* multiplier applied to int16 samples (ignored for f32)    */
  /* -- MelSpectrogram + AmplitudeToDB branch (ref: lid/audio_processor.py:72-105); all zero for the kaldi branch -- */
  int framing;       /* LIDFE_FRAMING_KALDI | LIDFE_FRAMING_CENTER               */
  int pad;           /* MelSpectrogram(pad=...): zeros added on both sides (CENTER framing only) */
  int log_kind;      /* LIDFE_LOG_NATURAL | LIDFE_LOG_DB10                       */
  float top_db;      /* LIDFE_POST_TOPDB: 80.0 in the reference                  */
  /* -- waveform dither inside the fused kernel (ref: lid/audio_processor.py:129 wav += 1e-5 * U[0,1); the kaldi call of
   *    the reference passes dither=0.0, ref: lid/audio_processor.py:57) -- */
  float dither;      /* 0 -> off (reference's wav2mel); > 0 -> x += dither * U[0,1) while the samples are staged,
                        Philox4x32-10 keyed by (seed, utterance, sample).  KALDI framing only                          */
  int window_type;   /* LIDFE_WINDOW_*: which window window_host holds (recorded and validated; the table itself is
                        built by the caller with the reference's fp32 arithmetic, ta: compliance/kaldi.py:86-113)      */
  unsigned long long seed;
} lidfe_config;

/* window kinds of torchaudio.compliance.kaldi._feature_window_function (ta: compliance/kaldi.py:86-113) plus the periodic
 * Hann of torch.stft (ref: lid/audio_processor.py:91-103) */
#define LIDFE_WINDOW_POVEY 0
#define LIDFE_WINDOW_HANNING 1
#define LIDFE_WINDOW_HAMMING 2
#define LIDFE_WINDOW_RECTANGULAR 3
#define LIDFE_WINDOW_BLACKMAN 4
#define LIDFE_WINDOW_HANN_PERIODIC 5

/* -- lifetime ------------------------------------------------------------------------------------- */

/*
 * Replaces the per-call table construction inside kaldi.fbank / kaldi.mfcc
 * (ta: compliance/kaldi.py:86-113 window, :436-511 mel banks, :648-666 DCT + lifter).
 * The caller builds the tables with the same fp32 host arithmetic as the reference and passes them in:
 *   window_host  [frame_len]
 *   melbank_host [n_mels][fft_len/2 + 1]   dense, row-major; sparsified inside
 *   dct_host     [n_mels][n_ceps]          or NULL when n_ceps == 0
 *   lifter_host  [n_ceps]                  or NULL (no liftering)
 * Uploads constant tables to the current device; allocates nothing else.
 */
int lidfe_create(lidfe_handle* out, const lidfe_config* cfg, const float* window_host,
                 const float* melbank_host, const float* dct_host, const float* lifter_host);
int lidfe_destroy(lidfe_handle h);

/* Number of frames.  KALDI framing (ta: compliance/kaldi.py:63-67): 1 + (n - frame_len) / frame_shift, or 0 when
 * n < frame_len.  CENTER framing (torch.stft): 1 + (n + 2 pad) / frame_shift, or 0 when n + 2 pad <= fft_len / 2
 * (reflect padding needs more samples than it mirrors; torch raises there).  Host helper, integer-exact. */
long long lidfe_num_frames(long long n_samples, const lidfe_config* cfg);

/* Output feature dimension: n_ceps if n_ceps > 0 else n_mels. */
int lidfe_out_dim(lidfe_handle h);

/*
 * Host-only helpers (no device needed): how lidfe_create turns the dense (n_mels x 257) bank into the kernel's
 * segment plan.  The banks on this path (Kaldi / HTK triangles) overlap only with their neighbours, so lane m % 16 of
 * band m / 16 walks the FFT bins between the centres of filters m and m+1 once, with two weights per bin (its own
 * down-slope, the next filter's up-slope; slot 0 also takes the bins below the first centre).  Outputs, per slot m:
 * first bin and length of that run, and the (possibly earlier) first power bin the lane reads so that the 16 lanes of
 * a band hit 16 distinct shared-memory bank pairs; band_taps_out[5] = steps per band of 16 slots.
 * LIDFE_E_MELBANK when a bin feeds more than two filters, or two that are not adjacent, or a row is empty.
 * lidfe_mel_plan_expand replays the plan into dense_out[n_mels * 257]: it must equal the input bank bit for bit.
 */
int lidfe_mel_plan(int n_mels, const float* melbank_host, int* first_bin_out, int* num_taps_out, int* start_out,
                   int* band_taps_out);
int lidfe_mel_plan_expand(int n_mels, const float* melbank_host, float* dense_out);

/* -- plan: the segment-offset table of one batch -------------------------------------------------- */

/*
 * Replaces MergedDataset.collate_fn's padding bookkeeping (ref: lid/raw_datasets.py:345-365) and the
 * per-utterance Python loop around wav2mel (ref: lid/raw_datasets.py:270-305).
 *   wav_offsets_host [B]  first sample of utterance i inside the packed waveform buffer (in samples)
 *   wav_lengths_host [B]  number of samples of utterance i  (>= frame_len, else LIDFE_E_SHORT)
 *   out_rows_host    [B]  output row of frame 0 of utterance i.  Packed: prefix sum of frame counts.
 *                         Padded (B, T_max, n_out): i * T_max.
 *   pad_rows_host    [B]  or NULL: rows [out_rows[i] + T_i, out_rows[i] + pad_rows[i]) are zero-filled by
 *                         the kernel (pad_sequence's zeros) -- no separate memset / pad pass.
 * Utterances whose offset is a multiple of 16 bytes are staged by TMA bulk copies; others fall back to
 * element loads (slower, same results).
 */
int lidfe_plan_create(lidfe_handle h, lidfe_plan* out, int B, const long long* wav_offsets_host,
                      const long long* wav_lengths_host, const long long* out_rows_host,
                      const long long* pad_rows_host);
/* The same without waiting: the table upload is ONE cudaMemcpyAsync from a pinned staging buffer on `stream`; memory
 * comes from the handle's pool (see Conventions).  This is what a training loop calls once per (ragged) batch. */
int lidfe_plan_create_async(lidfe_handle h, lidfe_plan* out, int B, const long long* wav_offsets_host,
                            const long long* wav_lengths_host, const long long* out_rows_host,
                            const long long* pad_rows_host, void* stream);
/* Returns the plan's memory to the handle's pool (no cudaFree; the pool is released by lidfe_destroy). */
int lidfe_plan_destroy(lidfe_plan p);
/* Pool bookkeeping (tests / monitoring): allocations made for plans since lidfe_create, and blocks currently free. */
int lidfe_pool_stats(lidfe_handle h, long long* blocks_allocated, long long* blocks_free);
long long lidfe_plan_total_frames(lidfe_plan p);
long long lidfe_plan_num_tiles(lidfe_plan p);
/* work items ("spans": runs of consecutive tiles of one utterance) the fused kernel's CTAs claim dynamically */
long long lidfe_plan_num_spans(lidfe_plan p);
/* frames of utterance i (host copy of what the kernel will produce) */
long long lidfe_plan_frames(lidfe_plan p, int i);

/* -- the hot path --------------------------------------------------------------------------------- */

/*
 * One fbank kernel for every cmvn_mode.  With LIDFE_CMVN_PER_UTT / LIDFE_POST_TOPDB it also hands each utterance's
 * statistics (sums / extrema) over to global memory, and a second kernel, cmvn_apply_kernel, normalises (clamps) the
 * rows in place: it reads them back, mostly out of L2, where the fbank kernel has just written them.
 * lidfe_set_precision changes which kernels this call launches: it mutates the handle and must not race with launches.
 * Replaces, for a whole batch in one call:
 *   wav2mel(x, use_kaildi=True)            ref: lid/audio_processor.py:8-69   (n_ceps == 0)
 *   torchaudio.compliance.kaldi.mfcc       ta: compliance/kaldi.py:669-813    (n_ceps > 0; not in the reference)
 *   spectrogram_augment(mask application)  ref: lid/audio_processor.py:225-227; ta: functional/functional.py:885-958
 *   CMVN                                   commented out at ref: lid/audio_processor.py:66-68 (our definition)
 *   collate_fn padding                     ref: lid/raw_datasets.py:347-350
 *
 *   wav_dev       packed samples (float32 or int16 per cfg.in_dtype)
 *   out_dev       [rows][out_ld] float32, out_ld >= n_out
 *   masks_dev     int32 [B][n_masks][4] = (t0, t1, f0, f1): frames [t0,t1) and dims [f0,f1) of utterance i are
 *                 set to 0.0 after normalisation; NULL / n_masks == 0 -> no masking.  The integer bounds are drawn
 *                 on the host from the same RNG stream as the reference, so application is bit-exact.
 *   cmvn_mode     LIDFE_CMVN_*
 *   stats_in_dev  double [2*n_out + 1] = sum_d, sumsq_d, count  (APPLY_GLOBAL), else NULL
 *   stats_out_dev double [2*n_out + 1] accumulated with atomics (ACCUM_GLOBAL), else NULL.  Caller zeroes it.
 * With ACCUM_GLOBAL masks are ignored (they are applied by lidfe_cmvn_apply after the all-reduce).
 */
int lidfe_featurize(lidfe_handle h, lidfe_plan p, const void* wav_dev, float* out_dev, long long out_ld,
                    const int* masks_dev, int n_masks, int cmvn_mode, const double* stats_in_dev,
                    double* stats_out_dev, void* stream);

/*
 * read_audio(normalize=True) + wav2mel in one call (ref: lid/audio_processor.py:108-122 then :8-69): same arguments as
 * lidfe_featurize, but wav_dev holds RAW samples (int16 PCM scaled by cfg.in_scale, or float32).  A statistics pre-pass
 * (wave_stages_kernel, mean and unbiased std per utterance) is followed by the fused kernel, which applies
 * (x - mean) / (std + 1e-6) while it stages each tile -- the raw samples are the only waveform bytes read or written.
 */
int lidfe_featurize_raw(lidfe_handle h, lidfe_plan p, const void* wav_dev, float* out_dev, long long out_ld,
                        const int* masks_dev, int n_masks, int cmvn_mode, const double* stats_in_dev,
                        double* stats_out_dev, void* stream);

/*
 * Second pass of global CMVN: feats = (feats - mean) / (std + 1e-9) in place, then masks.
 * stats_dev is the all-reduced [2*n_out + 1] vector.  (Global CMVN has no reference implementation.)
 */
int lidfe_cmvn_apply(lidfe_handle h, lidfe_plan p, float* feats_dev, long long ld, const int* masks_dev,
                     int n_masks, const double* stats_dev, void* stream);

/*
 * Standalone SpecAugment application (ref: lid/audio_processor.py:225-227; ta: functional/functional.py:885-958):
 * zero-fill frames [t0,t1) and dims [f0,f1) of every utterance of the plan, in place.  Used by the
 * single-utterance spectrogram_augment() wrapper; lidfe_featurize applies the same table in its epilogue.
 */
int lidfe_mask_apply(lidfe_handle h, lidfe_plan p, float* feats_dev, long long ld, const int* masks_dev, int n_masks,
                     void* stream);

/*
 * Waveform-level stages that precede framing, per utterance of the plan, float32 in -> float32 out
 * (out-of-place: wav_out_dev must not alias wav_in_dev; the reference's wav_augment mutates its input, the
 * Python wrapper restores that behaviour by copying back):
 *   normalize != 0 : normalize_wav  (x - mean) / (std + 1e-6), unbiased std     ref: lid/audio_processor.py:108-115
 *   dither   != 0  : x += dither * noise_dev[i]   (noise = the U[0,1) draw)     ref: lid/audio_processor.py:129
 *   preemph  != 0  : y[0] = x[0]; y[n] = x[n] - preemph * x[n-1]                ref: lid/audio_processor.py:131-134
 * noise_dev may be NULL when dither == 0.  Offsets/lengths are the plan's.
 */
int lidfe_wave_stages(lidfe_handle h, lidfe_plan p, const float* wav_in_dev, float* wav_out_dev, int normalize,
                      float dither, const float* noise_dev, float preemph, void* stream);
/* noise_dev == NULL with dither != 0: the noise is drawn on the device, Philox4x32-10 keyed by (cfg.seed, utterance,
 * sample) -- no host-drawn buffer crosses PCIe.  (noise_dev != NULL keeps bit parity with the reference's RNG stream.) */

/* Same stages fed with raw int16 PCM (what torchaudio.load decodes from a 16-bit wav before scaling by 1/32768,
 * ref: lid/audio_processor.py:118-122): x = (float)pcm * in_scale first.  Lets the host ship 2 bytes per sample. */
int lidfe_wave_stages_i16(lidfe_handle h, lidfe_plan p, const short* pcm_in_dev, float in_scale, float* wav_out_dev,
                          int normalize, float dither, const float* noise_dev, float preemph, void* stream);

/* -- measurement --------------------------------------------------------------------------------
 * Between lidfe_profile_begin and lidfe_profile_end every lidfe_featurize call brackets its fused fbank kernel with
 * a CUDA event pair on the launching stream (up to max_launches calls).  lidfe_profile_end synchronises on them and
 * returns the per-launch durations in milliseconds (bench.py's roofline leg).  Not thread-safe per handle. */
int lidfe_profile_begin(lidfe_handle h, int max_launches);
/* bracket only every stride-th call (default 1): an event record between two kernels costs a few microseconds */
int lidfe_profile_set_stride(lidfe_handle h, int stride);
int lidfe_profile_end(lidfe_handle h, float* ms_host, int capacity, int* n_out);

/* -- misc ----------------------------------------------------------------------------------------- */
/* -- polyphase sinc resampler: the DataProcessor in front of the models ------------------------------
 * Replaces torchaudio.transforms.Resample(orig_freq, 16000) as constructed by the reference for 22.05 and 44.1 kHz
 * input (ref: lid/ConformerLangModel.py:131-169 -> ta: transforms/_transforms.py Resample, functional/functional.py
 * _get_sinc_resample_kernel / _apply_sinc_resample_kernel).  kernel_host[new/g][taps] is the FIR bank exactly as
 * torchaudio builds it (g = gcd, taps = 2 * width + orig / g); the caller computes it with the same torch expressions
 * (speech_lid_b200.tables.sinc_resample_kernel).  Output sample j of an utterance of n samples exists for
 * j < ceil(new * n / orig); out_len_dev[i] may ask for fewer (the reference crops to int(percent * padded length)). */
typedef struct lidfe_resampler_s* lidfe_resampler;
int lidfe_resampler_create(lidfe_resampler* out, int orig_freq, int new_freq, const float* kernel_host, int taps, int width);
int lidfe_resampler_destroy(lidfe_resampler r);
long long lidfe_resample_out_len(lidfe_resampler r, long long n_in);
int lidfe_resample(lidfe_resampler r, int B, const float* in_dev, const long long* in_off_dev, const long long* in_len_dev,
                   float* out_dev, const long long* out_off_dev, const long long* out_len_dev, long long max_out_len,
                   void* stream);

/* -- the wav2vec-exp FBank variant (ref: wav2vec-exp/s3prl_model.py:174-204) --------------------------------------------
 * lidfe_wgemm_create: the resampler kernels as a general windowed GEMM,
 *     out[f * n_rows + p] = sum_k bank_host[p][k] * xpad[f * hop - left_pad + k]     (n_rows even, run with lidfe_resample,
 *     out_len = frames * n_rows).  The FBank variant passes a windowed DFT basis: row 2 b = w[k] cos(2 pi b k / n_fft),
 *     row 2 b + 1 = -w[k] sin(...), hop = n_fft / 2, left_pad 0 (torch.stft center=False), rows padded with zeros to a
 *     count the tensor-core kernel tiles (speech_lid_b200.S3prlFBank does this).
 * lidfe_stft_mel_db: rows of that GEMM -> |X|^2 -> mel (melT_dev[n_mels][n_bins], non-zero range mel_lo/mel_hi per filter:
 *     F.melscale_fbanks transposed) -> 10 log10(max(., amin)) into out_dev[(out_row[i] + t) * n_mels + m]; normalize != 0:
 *     then (x - mean) / (std + 1e-9) with one mean / unbiased std per utterance (stats_dev[B][2] is workspace). */
int lidfe_wgemm_create(lidfe_resampler* out, int hop, int n_rows, const float* bank_host, int taps, int left_pad);
int lidfe_stft_mel_db(const float* g_dev, const long long* g_off_dev, const long long* frames_dev, int B, long long max_frames,
                      int nw, const float* melT_dev, const int* mel_lo_dev, const int* mel_hi_dev, int n_bins, int n_mels,
                      float amin, float* out_dev, const long long* out_row_dev, double* stats_dev, int normalize, void* stream);

/* Arithmetic mode of lidfe_featurize on this handle.  0 (default): the fast fp32 kernels.  1: "precise" -- the reference's
 * formula (ref: lid/audio_processor.py:41-69 -> ta: compliance/kaldi.py:183-217, 514-645, 648-813) evaluated in float64
 * from the samples to the logarithm (through DCT + lifter for MFCC) on the same fp32 tables, rounded once at the store:
 * within half an ulp of the fp64 truth, i.e. at least as close to it as the reference's own fp32 result on every mel bin
 * (SURVEY.md 8c metric iv).  About 3 x the time of the fast path.  Scope: both framings (the Kaldi call and the default
 * MelSpectrogram + AmplitudeToDB branch, ref: lid/audio_processor.py:72-105), both logs, every cmvn mode; no in-kernel
 * dither (LIDFE_E_CONFIG); lidfe_featurize_raw is not served (LIDFE_E_ARG).
 * No allocation, no synchronisation: the mode reads the handle's existing tables. */
int lidfe_set_precision(lidfe_handle h, int precise);

/* FP32 ceiling of the device, measured: a dependent-free FFMA loop on every SM for about `ms_budget` milliseconds.
 * Writes the achieved TFLOP/s (2 flops per FFMA) -- bench.py reports the kernel against this, not against a data sheet. */
int lidfe_fp32_probe(float ms_budget, double* tflops_out, void* stream);

/* Host-side gather of a batch into the packed layout a plan describes (replaces the host half of the reference's
 * collate, ref: lid/raw_datasets.py:345-351, whose pad_sequence copies every waveform once as well): utterance i
 * (lengths[i] elements of elem_bytes = 4 for float32 or 2 for int16 PCM, at src_host[i]) is copied to
 * dst_host + offsets[i] * elem_bytes; the alignment gaps and the tail up to total_elems are zeroed.  The byte range is
 * split over `threads` host threads (0 = hardware concurrency, at most 32).  dst_host is normally pinned memory that
 * the caller then ships with one cudaMemcpyAsync.  No CUDA call is made. */
int lidfe_pack_host(void* dst_host, const void* const* src_host, const long long* offsets, const long long* lengths,
                    int B, int elem_bytes, long long total_elems, int threads);

/* The same gather for sources that already sit in pinned host memory (a DataLoader with pin_memory=True): no staging
 * copy; the data goes straight to dst_dev + offsets[i] * elem_bytes on `stream`.  When every source is 16-byte aligned and
 * mapped into the device's address space (cudaHostAlloc'ed memory under UVA: what torch's pin_memory() hands out) the SMs
 * read the host buffers themselves -- one gather kernel per <= 120 utterances; 256 utterances of ~0.7 MB: 3.6 ms against
 * 4.5 ms for as many cudaMemcpyAsync calls, whose per-copy set-up leaves the link idle --; otherwise one cudaMemcpyAsync per
 * utterance.  The gaps are not written (the kernels never read them).  The caller keeps the sources alive until the
 * stream has passed this point. */
int lidfe_h2d_gather(void* dst_dev, const void* const* src_host, const long long* offsets, const long long* lengths,
                     int B, int elem_bytes, void* stream);

const char* lidfe_strerror(int rc);
int lidfe_abi_version(void);
/* kernels launched by this library in this process so far (bench.py reports it as gpu_launches) */
long long lidfe_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* LIDFE_H_ */
