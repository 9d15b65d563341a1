#!/usr/bin/env python
"""bench.py -- audio-seconds/second of the speech-lid front-end hot path on B200.

Workload (BASELINE.json configs[1]): 80-dim Kaldi fbank + SpecAugment (2 time + 2 frequency masks) +
per-utterance CMVN on a batch of 256 x 8-s 16 kHz utterances per GPU (synthetic, seeded).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One JSON line on rank 0.  `value` = whole-job audio-s/s with inputs resident in HBM (weak scaling: every rank
processes its own 256-utterance batch; utterances are independent, no data-path collective).  `e2e` = the same
metric through the public host API with pinned HOST buffers (H2D of the waveforms and D2H of the features inside
the timed region).  `roofline` describes the dominant kernel (the fused fbank kernel, which since round 2 also
normalises: the step is ONE kernel) from CUDA-event timings inside the timed region, against the binding bound --
FP32 flops, whose ceiling is measured in the same run by an FFMA probe -- with the HBM figure beside it.
`sustained` repeats the step for >= 2 s with the clocks sampled throughout.  `cfg4` (every N, strong scaling) is
BASELINE config 4: 10 000 utterances of 1-20 s (seed 3) packed by an offset table, LPT-sharded by utterance,
global CMVN = accumulate -> ONE all-reduce of 161 doubles -> apply, the all-reduce inside the timed region.
`e2e_ragged` feeds a different ragged batch every step through DeviceCollate (plan creation inside the timed
region).  `cpu_baseline` = the reference path (torchaudio's kaldi.fbank + masking transforms, as
lid/audio_processor.py calls them) on the box's host cores (rank 0, N=1 only), all cores and one core.
--impl reference times that CPU path as the reference arm.

--dump-outputs DIR writes what the headline's last timed step returned (rank 0): DIR/features.npy, float32
[128, 798, 80], the features of a fixed seeded sample of 128 of the batch's 256 utterances (the whole batch is 65 MB).
The inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B_UTTS = 256
N_SAMPLES = 128000
SR = 16000
N_MELS = 80
T_MASK, F_MASK, MASK_TIMES = 0.05, 27, 2
AUDIO_S_PER_BATCH = B_UTTS * N_SAMPLES / SR          # 2048
ALG_BYTES_PER_FRAME = 160 * 4 + N_MELS * 4             # SURVEY.md §8(d): 640 B in + 320 B out per 10-ms frame
ALG_FLOP_PER_FRAME = 15.0e3                            # SURVEY.md §8(d)
METRIC = "audio-sec/sec 80-dim fbank+SpecAugment+CMVN"
WORKLOAD = "cfg2: 80-dim kaldi fbank + SpecAugment(t_mask=0.05,f_mask=27,x2) + per-utterance CMVN, 256 x 8-s utterances per GPU"
DUMP_UTTS, DUMP_SEED = 128, 0


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path, one worker process per host core
# ------------------------------------------------------------------------------------------------
def _cpu_worker_init():
    import torch
    torch.set_num_threads(1)


def _reference_path():
    """(wav2mel, augment, name): the reference's per-utterance calls.  With torchaudio importable these ARE the library
    calls lid/audio_processor.py makes (ref: lid/audio_processor.py:54-65, 225-227); otherwise the oracle's restatement
    of them with the same torch CPU ops."""
    import torch
    from oracle import frontend_oracle as O
    try:
        import torchaudio
        from torchaudio.compliance import kaldi as K
        tm = {}

        def wav2mel(x):
            f = K.fbank(x, num_mel_bins=N_MELS, dither=0.0, frame_length=25, frame_shift=10,
                        preemphasis_coefficient=1.0, sample_frequency=SR)
            return f.transpose(0, 1).unsqueeze(0)

        def augment(spec):
            T = spec.shape[-1]
            for _ in range(MASK_TIMES):
                key = int(T * T_MASK)
                if key not in tm:
                    tm[key] = torchaudio.transforms.TimeMasking(key)
                spec = tm[key](spec)
                spec = tm.setdefault("f", torchaudio.transforms.FrequencyMasking(F_MASK))(spec)
            return spec
        return wav2mel, augment, "torchaudio %s kaldi.fbank + Time/FrequencyMasking" % torchaudio.__version__
    except Exception:
        gen = torch.Generator().manual_seed(7)
        return (O.wav2mel_kaldi,
                lambda spec: O.spectrogram_augment(spec, T_MASK, F_MASK, MASK_TIMES, generator=gen),
                "oracle restatement (torchaudio not importable)")


def _cpu_worker(args):
    """Reference path for a share of the batch, exactly as MergedDataset.__getitem__ runs it per utterance
    (ref: lid/raw_datasets.py:270-305): wav2mel(use_kaildi=True) -> [our CMVN] -> spectrogram_augment."""
    import torch
    from oracle import frontend_oracle as O
    seed, n_utts, n_samples, reps = args
    g = torch.Generator().manual_seed(seed)
    wavs = [O.normalize_wav(torch.randn(1, n_samples, generator=g)) for _ in range(n_utts)]
    torch.manual_seed(seed + 1)
    wav2mel, augment, _ = _reference_path()
    times = []
    acc = 0.0
    for _ in range(reps):
        t0 = time.perf_counter()
        for w in wavs:
            spec = wav2mel(w)                                                    # (1, 80, T)
            feat = O.cmvn_per_utt(spec[0].T)                                     # (T, 80)
            spec = augment(feat.T.unsqueeze(0))
            acc += float(spec[0, 0, 0])
        times.append(time.perf_counter() - t0)
    return times, acc


def run_cpu_arm(steps, warmup, n_utts_total=B_UTTS, n_samples=N_SAMPLES):
    """Returns (audio_s_per_s, seconds_per_step, cores).  Every step is the full 256 x 8-s batch split over all
    host cores; per-step time = the slowest worker's time for that step (workers run concurrently)."""
    import multiprocessing as mp
    cores = max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    workers = min(cores, n_utts_total)
    share = [n_utts_total // workers + (1 if i < n_utts_total % workers else 0) for i in range(workers)]
    ctx = mp.get_context("spawn")
    t_wall0 = time.perf_counter()
    with ctx.Pool(workers, initializer=_cpu_worker_init) as pool:
        res = pool.map(_cpu_worker, [(1000 + i, share[i], n_samples, steps + warmup) for i in range(workers)])
    wall = time.perf_counter() - t_wall0
    per_step = [max(r[0][s] for r in res) for s in range(warmup, warmup + steps)]
    sec = sum(per_step) / len(per_step)
    audio_s = n_utts_total * n_samples / SR
    return audio_s / sec, sec, workers, wall


def run_cpu_single_core(n_utts=4, n_samples=N_SAMPLES):
    """The same per-utterance path on ONE core (torch threads = 1), a few utterances: audio-s/s."""
    import torch
    torch.set_num_threads(1)
    times, _ = _cpu_worker((999, n_utts, n_samples, 2))
    return n_utts * n_samples / SR / times[1]


_JSON_OUT = None


def keep_stdout_clean():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on the first
    collective): file descriptor 1 is pointed at stderr for the whole run and the line goes out through a private
    duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def dump_pick():
    """The utterances --dump-outputs keeps: a fixed seeded sample of DUMP_UTTS of the B_UTTS, in batch order."""
    import torch
    return torch.randperm(B_UTTS, generator=torch.Generator().manual_seed(DUMP_SEED))[:DUMP_UTTS].sort().values


def write_outputs(out_dir, arrays):
    """DIR/<name>.npy per array, float32 as computed."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().numpy())


def config_dict(world):
    """Identical in both arms."""
    return {"workload": WORKLOAD, "utterances_per_gpu": B_UTTS, "samples_per_utterance": N_SAMPLES,
            "frames_per_gpu_step": B_UTTS * (1 + (N_SAMPLES - 400) // 160),
            "parallelism": "utterance-sharded x%d" % world,
            "l2": "3 rotating input/output sets (196 MB per step > 126 MB L2)"}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU while the timed region runs (pynvml; nvidia-smi fallback)."""

    def __init__(self, index, period=0.002):
        self.index = index
        self.period = period
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._h = None

    def _decode(self, mask):
        nv = self._nv
        names = {"hw_slowdown": "nvmlClocksThrottleReasonHwSlowdown",
                 "hw_thermal_slowdown": "nvmlClocksThrottleReasonHwThermalSlowdown",
                 "sw_thermal_slowdown": "nvmlClocksThrottleReasonSwThermalSlowdown",
                 "sw_power_cap": "nvmlClocksThrottleReasonSwPowerCap",
                 "hw_power_brake": "nvmlClocksThrottleReasonHwPowerBrakeSlowdown"}
        for k, attr in names.items():
            bit = getattr(nv, attr, None)
            if bit is not None and (mask & bit):
                self.reasons.add(k)

    def sample_once(self):
        if self._h is None:
            return
        try:
            self.samples.append(self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM))
            self._decode(self._nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
        except Exception:
            pass

    def _loop(self):
        while not self._stop.is_set():
            self.sample_once()
            self._stop.wait(self.period)

    def start(self):
        if self._h is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()
        if self._h is None:      # fallback: one nvidia-smi query right after the region
            try:
                import subprocess
                out = subprocess.check_output(
                    ["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                     "--format=csv,noheader,nounits"], timeout=20).decode().strip().split(",")
                self.samples.append(int(out[0]))
                self.max_mhz = int(out[1])
            except Exception:
                pass
        return {"sm_mhz": (statistics.median(self.samples) if self.samples else None),
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def pipe_floors(frames, sms, mhz):
    """Per-launch floors of the two SM pipes the fused kernel loads most, from the per-quad (4-frame) counts of
    profiles/r2_fbank_warp_ncu_summary.txt: 480 shared-memory wavefronts (1 per clock and SM), 615 packed f32x2 operations
    at 2 issue cycles each + 190 scalar ones spread over the 4 sub-partitions."""
    quads_per_sm = frames / 4.0 / sms
    return {"smem_data_pipe": round(quads_per_sm * 480.0 / mhz, 1),
            "fma_pipe_instruction_mix": round(quads_per_sm * (615.0 * 2.0 + 190.0) / 4.0 / mhz, 1),
            "source": "profiles/r2_fbank_warp_ncu_summary.txt (per quad: 480 wavefronts, 615 f32x2 + 190 scalar FP instructions)"}


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)

    import speech_lid_b200 as lid
    fe = lid.FrontEnd(n_mels=N_MELS, device=dev)
    lib = lid.load_library()
    plan = fe.make_plan([N_SAMPLES] * B_UTTS, padded=True)
    frames_per_step = plan.total_frames

    # resident inputs: NBUF rotating sets so that no step finds its waveforms or its output lines in L2
    NBUF = 3
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    ins, outs = [], []
    for _ in range(NBUF):
        w = torch.randn(B_UTTS, N_SAMPLES, device=dev, generator=g)
        w = (w - w.mean(1, keepdim=True)) / (w.std(1, keepdim=True) + 1e-6)      # normalize_wav'ed, as the reference feeds it
        ins.append(w.reshape(-1).contiguous())
        outs.append(torch.empty(B_UTTS, plan.t_max, N_MELS, device=dev))
    torch.manual_seed(1234)
    masks = lid.draw_masks(plan.frames, N_MELS, T_MASK, F_MASK, MASK_TIMES).to(dev)

    def step(i):
        fe.featurize_packed(ins[i % NBUF], plan, out=outs[i % NBUF], masks=masks, cmvn="utt")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(args.warmup):
        step(i)
    barrier()

    nvml_index = torch.cuda._get_nvml_device_index(dev) if hasattr(torch.cuda, "_get_nvml_device_index") else local_rank
    sampler = ClockSampler(nvml_index)
    prof_stride = 4 if args.steps >= 16 else 1     # sample the kernel timing: an event record between kernels costs ~us
    fe.profile_begin(args.steps, stride=prof_stride)
    launches0 = lib.lidfe_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    barrier()
    ev0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    ev1.record()
    sampler.sample_once()
    barrier()
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    launches = lib.lidfe_launch_count() - launches0
    kernel_ms = fe.profile_end()
    dump = None
    if args.dump_outputs and rank == 0:
        # taken now: the sections below overwrite the rotating output sets
        dump = {"features": outs[(args.warmup + args.steps - 1) % NBUF].index_select(0, dump_pick().to(dev)).cpu()}

    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = world * AUDIO_S_PER_BATCH / (ms_step * 1e-3)

    # ---- sustained: the same step back to back for >= 2 s, clocks sampled throughout (the headline region lasts a few
    #      tens of ms; this shows whether the figure holds once the boost budget is spent) --------------------------
    sus_steps = max(args.steps, int(2.2 / (ms_step * 1e-3)))
    sus_sampler = ClockSampler(nvml_index, period=0.01)
    barrier()
    sus_sampler.start()
    ev0.record()
    for i in range(sus_steps):
        step(i)
    ev1.record()
    barrier()
    sus_clocks = sus_sampler.stop()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sus_ms = float(t.item())
    sustained = {"value": round(world * AUDIO_S_PER_BATCH * sus_steps / (sus_ms * 1e-3), 1), "unit": "audio-s/s",
                 "steps": sus_steps, "seconds": round(sus_ms * 1e-3, 3), "clocks": sus_clocks}

    # ---- cold vs warm L2 (SURVEY.md 8d): the headline rotates 3 input/output sets (588 MB, nothing of a step's data is in
    #      L2 when it starts); here ONE set is re-used every step, so whatever of its 131 MB of waveforms / 65 MB of
    #      features survives in the 126 MB L2 is found there ---------------------------------------------------------
    warm_steps = max(20, min(args.steps, 100))
    for _ in range(3):
        step(0)
    barrier()
    ev0.record()
    for _ in range(warm_steps):
        step(0)
    ev1.record()
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    warm_ms = float(t.item()) / warm_steps
    l2_pair = {"cold_ms_per_step": round(ms_step, 5), "warm_ms_per_step": round(warm_ms, 5),
               "warm_value": round(world * AUDIO_S_PER_BATCH / (warm_ms * 1e-3), 1), "unit": "audio-s/s",
               "note": "cold = the headline (3 rotating sets, 588 MB); warm = one 196 MB set re-used every step against 126 MB of L2"}

    # ---- e2e: public host API, pinned host buffers, H2D + kernels + D2H per step --------------------------
    host_in = torch.empty(B_UTTS * N_SAMPLES, dtype=torch.float32).pin_memory()
    host_in.copy_(ins[0].cpu())
    host_out = torch.empty(B_UTTS, plan.t_max, N_MELS, dtype=torch.float32).pin_memory()
    host_masks = masks.cpu().pin_memory()

    e2e_chunks = int(os.environ.get("LIDFE_E2E_CHUNKS", "8"))

    def e2e_step():
        fe.featurize_host(host_in, plan, host_out, masks=host_masks, cmvn="utt", chunks=e2e_chunks)

    e2e_steps = max(3, min(args.steps, 20))
    E2E_BLOCKS = 3

    def timed_blocks(step_fn, n_steps=e2e_steps):
        """Seconds per step: median over E2E_BLOCKS blocks of n_steps steps (the PCIe link is shared with whatever else
        runs on the host; one disturbed block would otherwise decide the number)."""
        for _ in range(2):
            step_fn()
        secs = []
        for _ in range(E2E_BLOCKS):
            barrier()
            t0 = time.perf_counter()
            for _ in range(n_steps):
                step_fn()
            torch.cuda.synchronize(dev)
            secs.append((time.perf_counter() - t0) / n_steps)
        return sorted(secs)[len(secs) // 2]

    def over_ranks(sec):
        tt = torch.tensor([sec], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    e2e_value = world * AUDIO_S_PER_BATCH / over_ranks(timed_blocks(e2e_step))
    h2d = host_in.numel() * 4 + host_masks.numel() * 4
    d2h = host_out.numel() * 4

    # informational: the same step fed with raw int16 PCM (2 B/sample over PCIe) into an int16 front-end: 1/32768
    # scaling + normalize_wav are fused into the kernel's sample load (row f2; statistics pre-pass + ONE fused kernel).
    # NOT the headline e2e: the reference's wav2mel boundary takes float32 waveforms.
    fe16 = lid.FrontEnd(n_mels=N_MELS, device=dev, in_dtype=torch.int16, in_scale=1.0 / 32768.0)
    plan16 = fe16.make_plan([N_SAMPLES] * B_UTTS, padded=True)
    host_pcm = (ins[0].cpu() * 3000.0).clamp(-32768, 32767).to(torch.int16).pin_memory()

    def pcm_step():
        fe16.featurize_host(host_pcm, plan16, host_out, masks=host_masks, cmvn="utt", chunks=e2e_chunks)

    pcm_value = world * AUDIO_S_PER_BATCH / over_ranks(timed_blocks(pcm_step))

    # ---- e2e with a DIFFERENT ragged batch every step through DeviceCollate (cfg4-like lengths, B = 256): plan creation
    #      (host-side fill + one async copy from the handle's pool), packing, H2D, the kernel and a D2H read of the
    #      result are all inside the timed region (ref: lid/raw_datasets.py:345-365 -- every real batch has its own
    #      length signature) ------------------------------------------------------------------------------------
    gl = torch.Generator().manual_seed(77 + rank)
    n_rag = 6
    rag_batches = []
    for _ in range(n_rag):
        lens = torch.randint(16000, 320001, (B_UTTS,), generator=gl).tolist()
        items = [(torch.randn(n, generator=gl).pin_memory(), torch.zeros(3, dtype=torch.long), "p", "a") for n in lens]
        rag_batches.append((items, sum(lens) / SR))
    collate = lid.DeviceCollate(fe, {"a": 0}, train=True, t_mask=T_MASK, f_mask=F_MASK, mask_times=MASK_TIMES, cmvn="utt")
    rag_state = {"i": 0, "audio": 0.0}

    def ragged_step():
        items, audio = rag_batches[rag_state["i"] % n_rag]
        rag_state["i"] += 1
        rag_state["audio"] += audio
        feats = collate(items)[0]
        float(feats[0, 0, 0])          # D2H read of the step's result

    for _ in range(n_rag):
        ragged_step()                  # warm the plan pool / allocator
    torch.cuda.synchronize(dev)
    rag_state["audio"] = 0.0
    barrier()
    t0 = time.perf_counter()
    for _ in range(2 * n_rag):
        ragged_step()
    torch.cuda.synchronize(dev)
    rag_sec = over_ranks(time.perf_counter() - t0)
    ta = torch.tensor([rag_state["audio"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ta)
    ragged = {"value": round(float(ta.item()) / rag_sec, 1), "unit": "audio-s/s", "steps": 2 * n_rag,
              "utterances_per_step": B_UTTS, "lengths": "U[1 s, 20 s], a new draw every step",
              "note": "DeviceCollate: H2D first (pinned items: zero-copy gather kernel, the SMs read the host buffers), plan + mask draw under it, fused kernels, D2H read, per step"}

    cfg4 = run_cfg4(lid, fe, dev, rank, world, barrier)

    # ---- precise mode (rank 0, N = 1; informational): the same cfg2 step through the float64 kernel
    #      (FrontEnd(precise=True) -> lidfe_set_precision -> fbank_precise_kernel), the arithmetic under which SURVEY.md 8(c)
    #      metric (iv) holds unrelaxed (tests/test_gpu_precise.py); device-resident like `value`, and end to end through
    #      featurize_host like `e2e` (where PCIe, not the kernel, sets the pace) -----------------------------------------
    precise = None
    if world == 1:
        fep = lid.FrontEnd(n_mels=N_MELS, device=dev, precise=True)
        planp = fep.make_plan([N_SAMPLES] * B_UTTS, padded=True)
        for i in range(3):
            fep.featurize_packed(ins[i % NBUF], planp, out=outs[i % NBUF], masks=masks, cmvn="utt")
        p_steps = max(5, min(args.steps, 30))
        barrier()
        ev0.record()
        for i in range(p_steps):
            fep.featurize_packed(ins[i % NBUF], planp, out=outs[i % NBUF], masks=masks, cmvn="utt")
        ev1.record()
        barrier()
        p_ms = ev0.elapsed_time(ev1) / p_steps

        def precise_e2e_step():
            fep.featurize_host(host_in, planp, host_out, masks=host_masks, cmvn="utt", chunks=e2e_chunks)

        p_e2e = AUDIO_S_PER_BATCH / timed_blocks(precise_e2e_step, n_steps=max(3, min(args.steps, 10)))
        precise = {"value": round(AUDIO_S_PER_BATCH / (p_ms * 1e-3), 1), "unit": "audio-s/s", "ms_per_step": round(p_ms, 5),
                   "steps": p_steps, "e2e": round(p_e2e, 1), "dtype": "f64 internally, one rounding to f32 at the store",
                   "slowdown_vs_fast": round(p_ms / ms_step, 2),
                   "note": "informational: lidfe_set_precision(h, 1); parity metric (iv) of SURVEY.md 8(c) holds unrelaxed in this mode"}

    # ---- cfg5 (rank 0, N = 1): features feeding the reference's Conformer forward on the device, when the model files
    #      have been staged (baseline/_ref, see __graft_entry__.stage_reference_model)
    cfg5 = None
    if world == 1:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import cfg5_device
            cfg5 = cfg5_device.run(B=128, n_check=8, steps=3)
            if cfg5 is not None:
                cfg5.pop("consumer", None)
            else:
                cfg5 = {"unavailable": "the reference's model source is not staged in baseline/_ref/lid"}
        except Exception as ex:       # the consumer is not the product: never let it take the bench line down
            cfg5 = {"unavailable": "%s: %s" % (type(ex).__name__, ex)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak_src = "fallback (B200_PROFILING.md)"
    hbm_peak = 6650.0
    if os.path.exists(peaks_path):
        try:
            hbm_peak = float(json.load(open(peaks_path))["hbm_gbs"])
            peak_src = "MEASURED_PEAKS.json"
        except Exception:
            pass
    k_ms = statistics.mean(kernel_ms) if kernel_ms else float("nan")
    alg_bytes = frames_per_step * ALG_BYTES_PER_FRAME
    hbm_achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    fp32_theory = sms * 128 * 2 * (clocks.get("sm_max_mhz") or 1965) * 1e6 / 1e12
    import ctypes
    tf = ctypes.c_double(0.0)
    lid._lib.check(lib.lidfe_fp32_probe(30.0, ctypes.byref(tf), torch.cuda.current_stream(dev).cuda_stream))
    fp32_peak = float(tf.value)                      # FFMA loop on every SM, measured in this run
    fp32_achieved = frames_per_step * ALG_FLOP_PER_FRAME / (k_ms * 1e-3) / 1e12
    hbm_floor_us = alg_bytes / (hbm_peak * 1e9) * 1e6
    fp32_floor_us = frames_per_step * ALG_FLOP_PER_FRAME / (fp32_peak * 1e12) * 1e6
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("fbank_kernel_dram_bytes_per_launch")
        except Exception:
            traffic = None
    # the bound that binds is the slower floor (SURVEY.md 8d): FP32 flops here (41-44 us vs 30 us of HBM time)
    fp32_binds = fp32_floor_us >= hbm_floor_us
    roofline = {"bound": "fp32" if fp32_binds else "hbm", "kernel": "fbank_warp_kernel<float,1,true> (framing + FFT + mel + log + per-utterance sums; followed by cmvn_apply_kernel: 2 launches per step)",
                "achieved": round(fp32_achieved if fp32_binds else hbm_achieved, 2),
                "peak": round(fp32_peak if fp32_binds else hbm_peak, 2),
                "peak_source": "in-run FFMA probe (lidfe_fp32_probe)" if fp32_binds else peak_src,
                "unit": "TFLOP/s" if fp32_binds else "GB/s",
                "frac": round((fp32_achieved / fp32_peak) if fp32_binds else (hbm_achieved / hbm_peak), 4),
                "traffic": traffic, "kernel_ms": round(k_ms, 5), "kernel_share_of_step": round(k_ms / ms_step, 3),
                "kernel_timing": "CUDA event pair around every %d-th launch of the timed region (%d samples)" % (prof_stride, len(kernel_ms)),
                "alg_flop_per_launch": frames_per_step * ALG_FLOP_PER_FRAME, "alg_bytes_per_launch": alg_bytes,
                "floors_us": {"fp32": round(fp32_floor_us, 1), "hbm": round(hbm_floor_us, 1)},
                # what actually binds (ncu counters of the committed capture, scaled to this launch and the max clock): the
                # shared-memory data pipe delivers one 128-byte wavefront per clock and SM; the FFT is add-dominated, so its
                # 15 kflop per frame take more FMA-pipe cycles than as many flops of pure FFMA would
                "pipe_floors_us": pipe_floors(frames_per_step, sms, clocks.get("sm_max_mhz") or 1965),
                "fp32": {"achieved_tflops": round(fp32_achieved, 2), "peak_tflops_measured": round(fp32_peak, 2),
                         "peak_tflops_theoretical_at_max_clock": round(fp32_theory, 1),
                         "frac_of_measured": round(fp32_achieved / fp32_peak, 4),
                         "frac_at_max_clock": round(fp32_achieved / fp32_theory, 4),
                         "note": "algorithmic 15.0 kflop/frame (SURVEY.md 8d)"},
                "hbm": {"achieved_gbs": round(hbm_achieved, 1), "peak_gbs": hbm_peak, "peak_source": peak_src,
                        "frac": round(hbm_achieved / hbm_peak, 4)}}

    cpu = None
    if world == 1 and not args.no_cpu:
        v, sec, cores, wall = run_cpu_arm(steps=1, warmup=1)
        single = run_cpu_single_core()
        cpu = {"value": round(v, 1), "unit": "audio-s/s", "cores": cores, "kind": "port",
               "single_core": round(single, 1),
               "sample": "1 timed pass (after 1 warm-up) of the full 256 x 8-s batch, %s + CMVN, one process per core, "
                         "torch threads=1; %.1f s wall incl. start-up; single_core = 4 x 8-s utterances on one core"
                         % (_reference_path()[2], wall)}

    line = {"metric": METRIC, "value": round(value, 1), "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 5), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(world),
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 1), "unit": "audio-s/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "blocks": E2E_BLOCKS,
                    "agg": "median block", "pipeline_chunks": e2e_chunks},
            "e2e_int16_pcm": {"value": round(pcm_value, 1), "unit": "audio-s/s", "h2d_bytes_per_step": host_pcm.numel() * 2,
                              "d2h_bytes_per_step": d2h,
                              "note": "informational: host ships int16 PCM; scaling + normalize_wav fused into the kernel's sample load"},
            "e2e_ragged": ragged,
            "sustained": sustained,
            "l2_cold_warm": l2_pair,
            "cfg4": cfg4,
            "cfg5": cfg5,
            "precise": precise,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu}
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_cfg4(lid, fe, dev, rank, world, barrier, n_utts=None, steps=3):
    """BASELINE config 4 (SURVEY.md 8d-4, 8e): 10 000 utterances of 1-20 s (seed 3), packed by an offset table, sharded by
    utterance with the deterministic LPT partition, generated on the device (seed 3000 + rank); per pass:
    featurize(global_accum) -> all_reduce(161 fp64) -> cmvn_apply + masks.  STRONG scaling: the 10 k utterances are the
    whole job at every N.  Returns the sub-record (same on every rank)."""
    import torch
    import torch.distributed as dist
    n_utts = int(os.environ.get("LIDFE_CFG4_UTTS", "10000")) if n_utts is None else n_utts
    g = torch.Generator().manual_seed(3)
    lengths = torch.randint(16000, 320001, (n_utts,), generator=g).tolist()
    shards = lid.lpt_partition(lengths, world)
    mine = [lengths[i] for i in shards[rank]]
    plan = fe.make_plan(mine, padded=False)
    gd = torch.Generator(device=dev).manual_seed(3000 + rank)
    packed = torch.randn(plan.total_samples, device=dev, generator=gd)
    torch.manual_seed(99 + rank)
    masks = lid.draw_masks(plan.frames, N_MELS, T_MASK, F_MASK, MASK_TIMES).to(dev)
    out = torch.empty(plan.rows, N_MELS, device=dev)
    stats = torch.zeros(2 * N_MELS + 1, dtype=torch.float64, device=dev)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def one_pass(timed=False):
        stats.zero_()
        if timed:
            evs[0].record()
        fe.featurize_packed(packed, plan, out=out, cmvn="global_accum", stats_out=stats)
        if timed:
            evs[1].record()
        lid.allreduce_stats(stats)
        if timed:
            evs[2].record()
        fe.cmvn_apply(out, plan, stats, masks=masks)
        if timed:
            evs[3].record()

    one_pass()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one_pass()
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    one_pass(timed=True)
    torch.cuda.synchronize(dev)
    split = torch.tensor([evs[0].elapsed_time(evs[1]), evs[1].elapsed_time(evs[2]), evs[2].elapsed_time(evs[3])],
                         dtype=torch.float64, device=dev)
    load = torch.tensor([float(sum(mine))], dtype=torch.float64, device=dev)
    lo, hi = load.clone(), load.clone()
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(split, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    total_frames = int(stats[2 * N_MELS].item())
    audio_s = sum(lengths) / SR
    rec = {"workload": "cfg4: %d utterances 1-20 s (seed 3) packed, LPT-sharded x%d, global CMVN: accumulate -> "
                       "all_reduce(161 fp64) -> apply+masks, all-reduce inside the timed region" % (n_utts, world),
           "scaling": "strong", "n_gpus": world, "value": round(audio_s / (float(ms.item()) * 1e-3), 1), "unit": "audio-s/s",
           "ms_per_pass": round(float(ms.item()), 3), "steps": steps, "audio_s": round(audio_s, 1), "total_frames": total_frames,
           "split_ms_max_over_ranks": {"accumulate_kernel": round(float(split[0]), 3), "all_reduce": round(float(split[1]), 3),
                                        "apply_kernel": round(float(split[2]), 3)},
           "lpt_imbalance": round(float(hi.item() / lo.item()), 5),
           "comm": "1 x all_reduce(SUM, float64[161]) per pass over NCCL" if world > 1 else "none (N=1 base of the strong-scaling series)"}
    del packed, out
    return rec


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps = max(1, args.steps)
    warmup = max(0, args.warmup)
    v, sec, cores, wall = run_cpu_arm(steps=steps, warmup=warmup)
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 1), "unit": "audio-s/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": round(sec * 1e3, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(world),
            "cpu_baseline": {"value": round(v, 1), "unit": "audio-s/s", "cores": cores, "kind": "port",
                             "sample": "every step = the full 256 x 8-s batch split over %d single-thread worker "
                                       "processes; per utterance: %s + CMVN" % (cores, _reference_path()[2])},
            "e2e": {"value": round(v, 1), "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the features of the last timed step (a fixed sample of the batch) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    keep_stdout_clean()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
