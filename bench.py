"""Benchmark of the magnitude -> phase -> waveform hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl phasegen|reference|torch_gpu] [--workload ...]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Headline workload (configs[1] of BASELINE.json): 256 synthetic 4 s / 44.1 kHz mono clips per GPU,
n_fft 1024, hop 256 (T = 696 frames after padding to a multiple of 8, N = 177,920 samples),
STFT -> U-Net (C = 512, random-init weights, per-clip train-mode norm statistics = the
demo.py batch-1 loop) -> ISTFT with peak normalisation.  One "step" = one pass over the
batch.  metric = audio-seconds processed per wall second, whole job (all ranks).

The ONE JSON line of the default run also carries, as extra keys (each its own measurement):
  parity                 measured in this run: clips of the timed 256-clip batch against the CPU oracle chain
  gpu_library_baseline   the same workload through stock torch (cuFFT + cuDNN) on the same GPU      (N = 1)
  train                  BASELINE config 3: train.py step, UNetModel(1024, 2048), batch 32/GPU, bf16, data-parallel
  single_clip            BASELINE config 1: one 4 s clip, batch 1, eager and as a CUDA graph          (N = 1)
  longform               BASELINE config 4: a 10-minute clip, windows sharded over the N ranks
`--workload train|single|longform` print one of these as its own line instead.
`--dump-outputs DIR` writes the waves the last timed step of the headline workload returned (see dump_outputs).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "unet-phasegen_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

SR, N_FFT, HOP, SECONDS = 44100, 1024, 256, 4.0
CLIPS_PER_GPU = 256
# Inference default: fp16 operand planes (11+11 significant bits), three products per MAC on the five small layers, two on
# d1/u2 (weights rounded to fp16), ONE on the last layer u1 (both operands rounded to 11 bits = the operand rounding of the
# TF32 pass BASELINE.json's config 2 names, at twice its tensor rate; u1's rounding error is amplified by no later layer).
# Measured in every run against the float64 oracle (`parity`): predicted phase ~5.6e-4 vs the 1e-3 bound; a single TF32
# pass over all layers measures 1.3e-3 (SURVEY.md 8d).  `f16mix` (two products on u1 too: 5.1e-4) and `bf16x3` (three
# everywhere: 9.6e-5) are timed and checked beside it.
DEFAULT_PRECISION = "f16mix1"
METRIC = "audio_seconds_per_second_mag_to_phase_to_wave"
UNIT = "audio-s/s"
DUMP_BYTES = 64 * 2 ** 20


def workload_geometry():
    from phasegen import synth
    T = synth.frames_for(SECONDS, SR, HOP)
    N = (T - 1) * HOP
    return T, N, N / SR


def dump_outputs(out_dir, audio):
    """Write the waves [B, N] one headline step returned, so that two builds can be compared output for output on the
    same seeded inputs: out_dir/audio.npy (float32 [k, N]) holds k evenly spaced clips of the batch (all of them when they
    fit), as many as keep the dump under DUMP_BYTES, and out_dir/audio_clips.npy (float64 [k]) their indices in the batch."""
    import numpy as np
    import torch
    B, N = audio.shape
    k = max(1, min(B, (DUMP_BYTES - 2 ** 20) // (4 * N)))
    idx = np.unique(np.linspace(0, B - 1, k).round().astype(np.int64))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "audio.npy"), audio[torch.from_numpy(idx).to(audio.device)].float().cpu().numpy())
    np.save(os.path.join(out_dir, "audio_clips.npy"), idx.astype(np.float64))


def unet_flops_per_clip(C, T, phase_only):
    """Algorithmic MACs*2 of the eight convolutions (SURVEY.md section 8a), per clip."""
    L1 = T // 2 + 1; L2 = L1 - 3; L3 = L2 // 2 - 2; L4 = (L3 - 1) // 2
    c2, c4 = 2 * C, 4 * C
    per_layer = {
        "d1": C * c2 * 32 * L1, "d2": c2 * c2 * 8 * L2, "d3": c2 * c2 * 8 * L3, "d4": c2 * c4 * 4 * L4,
        "u4": c4 * c2 * 5 * L4, "u3": c4 * c2 * 8 * L3, "u2": c4 * c2 * 8 * L2,
        "u1": c4 * (C if phase_only else c2) * 32 * L1,
    }
    return {k: 2 * v for k, v in per_layer.items()}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        return {}


class ClockSampler:
    """SM clock and throttle reasons sampled WHILE the timed region runs: an NVML polling thread (every 5 ms), or the
    `nvidia-smi -lms` recipe when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}   # nvmlClocksEventReason*

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.sm, self.mask, self.max_mhz, self._stop, self._thread, self.source = [], 0, None, False, None, None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if not uuid.startswith("GPU-") else uuid.encode())
        except Exception:                                        # noqa: BLE001 -- older torch / NVML: ordinal order
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def start(self):
        try:
            nv, h = self._nvml_handle()
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                while not self._stop:
                    try:
                        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                        self.mask |= int(reasons(h))
                    except Exception:                            # noqa: BLE001
                        pass
                    time.sleep(0.005)
            self._thread = threading.Thread(target=poll, daemon=True)
            self._thread.start()
            self.source = "nvml"
            return
        except Exception:                                        # noqa: BLE001 -- no NVML binding: fall back to nvidia-smi
            self._thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            self.source = "nvidia-smi -lms 25"
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        """Samples taken so far (call at the start of the timed region: `stop()` reports what came after)."""
        self._from = len(self.sm) if self._thread is not None else len(self.rows)

    def stop(self):
        start = getattr(self, "_from", 0)
        if self._thread is not None:
            self._stop = True
            self._thread.join(timeout=1.0)
            sm = self.sm[start:] or self.sm
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": [n for n in self.NAMES if self.mask & self.BITS[n]], "samples": len(sm), "source": self.source}
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        rows = self.rows[start:] or self.rows
        sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        reasons = [n for i, n in enumerate(self.NAMES) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": self.source}


class Dist:
    """Rank plumbing shared by every leg: barrier + synchronize on both sides of a timed region, CUDA events on the
    launch stream, max over ranks."""

    def __init__(self):
        import torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the phasegen path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        # run (and first-touch the pinned staging buffers) on the NUMA node of this rank's GPU; best effort
        from phasegen import hostmem
        self.host_binding = hostmem.bind_to_gpu_node(self.local) if os.environ.get("PG_NO_NUMA_BIND") != "1" else {"numa_node": None, "disabled": True}
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        import torch
        torch.cuda.synchronize()
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps, finish=None):
        """Total milliseconds of `steps` calls, max over ranks.  `finish` (optional) runs after the last call and before
        the closing event: it orders work the calls left on other streams onto the timed stream."""
        import torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def close(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ CPU reference arm
def cpu_reference_step(n_clips, seed=0, time_budget_s=None, mkldnn=False):
    """The reference's CPU path (oracle port: numpy STFT/ISTFT restating librosa + the reference
    U-Net arithmetic through torch CPU fp32 with oneDNN off, batch 1 per clip like demo.py:33-42)
    on `n_clips` clips of the bench workload.  Returns (seconds, clips done)."""
    import numpy as np
    import torch
    from oracle import stft_np, unet_torch
    from phasegen import synth
    T, N, _ = workload_geometry()
    C = N_FFT // 2
    torch.set_num_threads(os.cpu_count() or 1)
    sd = unet_torch.random_state_dict(C, seed=seed)
    waves = synth.synthetic_waves(n_clips, N, SR, seed=seed).numpy()
    t0 = time.perf_counter()
    done = 0
    for i in range(n_clips):
        S = stft_np.stft(waves[i], N_FFT, HOP)[1:]
        lm = np.log1p(np.abs(S)).astype(np.float32)
        out = unet_torch.unet_forward(sd, torch.from_numpy(lm)[None], torch.float32, per_clip_bn=True, mkldnn=mkldnn)[0].numpy()
        stft_np.generate_audio(stft_np.polar_to_complex(lm, out[:C]), SR, HOP, is_stft=True)
        done += 1
        if time_budget_s is not None and time.perf_counter() - t0 > time_budget_s:
            break
    return time.perf_counter() - t0, done


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    T, N, clip_s = workload_geometry()
    cores = os.cpu_count() or 1
    n = 2
    for _ in range(args.warmup):
        cpu_reference_step(1)
    times = []
    for _ in range(args.steps):
        dt, done = cpu_reference_step(n)
        times.append(dt / done)
    per_clip = statistics.mean(times)
    value = clip_s / per_clip
    # BASELINE.md section 4: the stock oneDNN-on time, for context only -- its fp32 transposed convolution is ~22 % wrong in
    # this image (SURVEY.md section 0), so it is NOT a valid baseline
    cpu_reference_step(1, mkldnn=True)
    dt_on, done_on = cpu_reference_step(n, mkldnn=True)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_clip * n * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{n} clips/step of the batched-inference workload (4 s @ 44.1 kHz, n_fft {N_FFT}, hop {HOP}, "
                                   f"T {T}, C {N_FFT // 2}), batch-1 per clip like demo.py",
                       "timing": "host perf_counter; CPU only"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{n} clips per step x {args.steps} steps, oracle port (numpy STFT/ISTFT + torch-CPU fp32 U-Net, oneDNN off)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "onednn_on_numerically_invalid": {"value": clip_s * done_on / dt_on, "unit": UNIT,
                                              "note": "same loop with oneDNN enabled; its k5/s2 transposed convolution is ~22 % wrong here: context only, not a baseline"},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ measured parity
def measure_parity(pipe, net, wave, clips):
    """Parity of THIS run: the full batch goes through the pipeline once more (same executors, same tile plans as the
    timed steps, intermediates kept), and the listed clips are compared with the float64 CPU oracle chain
    (numpy STFT restating librosa -> reference U-Net arithmetic, per-clip statistics -> numpy ISTFT + peak normalise)."""
    import numpy as np
    import torch
    from oracle import stft_np, unet_torch
    C = N_FFT // 2
    audio, logmag, phase = pipe(wave, return_intermediates=True)
    torch.cuda.synchronize()
    overflow = bool(pipe.range_overflow())
    bad = pipe.nonfinite_clips(wave.shape[0])
    sd = {k: v.detach().cpu() for k, v in net.model.state_dict().items()}
    rel = lambda a, b: float(np.linalg.norm(np.asarray(a, np.float64) - b) / np.linalg.norm(b))

    def snr_db(ref, est):
        g = np.dot(ref, est) / max(np.dot(est, est), 1e-300)
        return 10 * np.log10(np.sum(ref ** 2) / np.sum((ref - g * est) ** 2))
    worst = {"logmag_rel_l2": 0.0, "phase_rel_l2": 0.0, "wave_rel_l2": 0.0, "snr_db_delta": 0.0}
    t0 = time.perf_counter()
    for b in clips:
        w = wave[b].cpu().numpy().astype(np.float64)
        lm = np.log1p(np.abs(stft_np.stft(w, N_FFT, HOP)[1:]))
        out = unet_torch.unet_forward(sd, torch.from_numpy(lm)[None], torch.float64, per_clip_bn=True)[0].numpy()
        ref = stft_np.generate_audio(stft_np.polar_to_complex(lm, out[:C]), SR, HOP, is_stft=True)
        got = audio[b].cpu().numpy().astype(np.float64)
        worst["logmag_rel_l2"] = max(worst["logmag_rel_l2"], rel(logmag[b].cpu().numpy().T, lm))
        worst["phase_rel_l2"] = max(worst["phase_rel_l2"], rel(phase[b].cpu().numpy().T, out[:C]))
        worst["wave_rel_l2"] = max(worst["wave_rel_l2"], rel(got, ref))
        worst["snr_db_delta"] = max(worst["snr_db_delta"], abs(snr_db(w, got) - snr_db(w, ref)))
    ok = (worst["logmag_rel_l2"] < 1e-4 and worst["phase_rel_l2"] < 1e-3 and worst["snr_db_delta"] < 0.1 and not overflow and not bad)
    return {"measured_in_this_run": True, "clips_checked": list(clips), "of_batch": int(wave.shape[0]),
            "vs": "float64 CPU oracle chain (oracle/stft_np.py + oracle/unet_torch.py)", **worst,
            "bounds": {"logmag_rel_l2": 1e-4, "phase_rel_l2": 1e-3, "snr_db_delta": 0.1},
            "fp16_range_overflow": overflow, "nonfinite_clips": len(bad), "pass": bool(ok),
            "oracle_seconds": round(time.perf_counter() - t0, 1)}


# ------------------------------------------------------------------------------------------ training (config 3)
def synthetic_train_pairs(B, C, T, seed, device):
    """"MedleyDB-shaped" pairs (SURVEY.md section 8d): z = complex N(0,1) * sigma(f) with a 1/f tilt;
    ch0 = log1p|z|, ch1 = angle z -- what data.py:39-47 yields.  Channels-last [B, T, C]."""
    import torch
    g = torch.Generator().manual_seed(seed)
    sigma = 4.0 / (1.0 + torch.arange(C, dtype=torch.float32) / 32.0)
    re = torch.randn(B, T, C, generator=g) * sigma
    im = torch.randn(B, T, C, generator=g) * sigma
    return torch.log1p(torch.sqrt(re * re + im * im)).contiguous().to(device), torch.atan2(im, re).contiguous().to(device)


def train_leg(args, D, with_library_baseline=False):
    """BASELINE.json config 3: train.py step (forward, cos/sin/mag loss, backward, Adam), UNetModel(1024, 2048),
    128-frame pairs, batch 32 per GPU, bf16 tensor-core products with fp32 accumulation and fp32 master weights,
    data-parallel over NCCL: one gradient exchange per step (reduce-scatter + sharded Adam + all-gather of the bf16
    operand planes; PG_TRAIN_ALLREDUCE=1 selects all-reduce + replicated Adam)."""
    import torch
    import model as pg_model
    from phasegen import _lib
    from phasegen.train import HostBatchFeeder, TrainStep
    world, rank, dev = D.world, D.rank, D.dev
    C, T, B = args.train_c, 128, args.train_batch
    torch.manual_seed(1234)
    net = pg_model.UNetModel(C, 2 * C).to(dev)
    train_prec = "bf16x3" if args.train_fp32 else (args.train_precision or "bf16")
    shard = None if not os.environ.get("PG_TRAIN_ALLREDUCE") else False
    step = TrainStep(net, B, T, dev, precision=train_prec, shard_optimizer=shard)
    lm, ph = synthetic_train_pairs(B, C, T, 100 + rank, dev)
    host = [t.cpu().pin_memory() for t in (lm, ph)]
    W = max(args.warmup, 3)
    losses = []

    def step_resident():
        step(lm, ph)

    feeder = HostBatchFeeder(tuple(lm.shape), dev)
    loss_host = [torch.zeros(4).pin_memory() for _ in range(2)]
    loss_ev = [None, None]
    e2e_i = [0]

    def step_e2e():
        # the public host path: pinned host batch -> copy stream -> step; the loss comes back through a pinned
        # buffer and is read one step late, so neither copy stalls the GPU
        k = e2e_i[0] & 1
        if loss_ev[k] is not None:
            loss_ev[k].synchronize()
            losses.append(float(loss_host[k][0]))
        a, b = feeder.next()                                   # uploaded underneath the previous step
        l3 = step(a, b)
        feeder.done()
        feeder.prefetch(host[0], host[1])                      # the next step's batch: one H2D copy of the batch per step
        loss_host[k].copy_(l3, non_blocking=True)
        loss_ev[k] = torch.cuda.Event(); loss_ev[k].record()
        e2e_i[0] += 1

    sampler = ClockSampler(D.local)
    if rank == 0:
        sampler.start()
    for _ in range(W):
        step_resident()
    l0 = _lib.launches
    sampler.mark()
    ms = D.timed(step_resident, args.steps)
    launches = _lib.launches - l0
    clocks = sampler.stop() if rank == 0 else None
    feeder.prefetch(host[0], host[1])
    for _ in range(2):
        step_e2e()
    ms_e2e = D.timed(step_e2e, args.steps)
    value = world * B / (ms / args.steps / 1e3)
    e2e = world * B / (ms_e2e / args.steps / 1e3)
    flops = 3 * sum(unet_flops_per_clip(C, T, False).values()) - unet_flops_per_clip(C, T, False)["d1"]   # no dgrad for d1
    peaks = load_peaks()
    peak = peaks.get("bf16_tflops_sustained") or 1590.0
    achieved = flops * B / (ms / args.steps / 1e3) / 1e12
    line = {"metric": "train_samples_per_second", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": f"{train_prec}-fp32acc (fp32 master weights, fp32 Adam)", "data": "synthetic",
            "config": {"workload": f"train.py step: UNetModel({C},{2 * C}) on [B,2,{C},{T}] log-mag/phase pairs, batch {B}/GPU, "
                                   "forward + cos/sin/mag loss + backward + Adam(lr 1e-3)", "parallelism": f"dp{world}",
                       "gradient_exchange": ("none (one GPU)" if world == 1 else "NCCL reduce-scatter (bf16 gradients) -> Adam on 1/N of the "
                                             "parameters per rank -> all-gather of the bf16 operand planes" if step.sharded is not None
                                             else "NCCL all-reduce (bf16 gradients) + replicated Adam"),
                       "timing": "CUDA events on the launch stream, max over ranks", "l2_policy": "weights + optimizer state (>10 GB) exceed L2"},
            "e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": 2 * B * T * C * 4, "d2h_bytes_per_step": 16, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "whole step (conv_tc + wgrad_tc dominate)", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": None, "note": "algorithmic FLOPs per GPU: fwd + dgrad + wgrad of the 8 convolutions"},
            "loss_trace": losses[-3:]}
    del step, feeder, net
    torch.cuda.empty_cache()
    if with_library_baseline and world == 1:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import torch_baseline
        line["gpu_library_baseline"] = torch_baseline.train_baseline(C, T, B)
    return line


# ------------------------------------------------------------------------------------------ single clip (config 1)
def single_clip_leg(args, D, net):
    """BASELINE.json config 1 (demo.py:33-42): ONE 4 s clip, batch 1, device-resident; eager call and CUDA-graph
    replay.  Roofline: at batch 1 the U-Net is weight-bandwidth-bound (SURVEY.md section 8d), so the HBM figure is
    the weight-plane bytes one pass must read divided by the time."""
    import torch
    from phasegen import synth
    from phasegen.pipeline import PhaseGenPipeline
    from phasegen.unet import F16MIX_FAST_LAYERS
    T, N, clip_s = workload_geometry()
    C = N_FFT // 2
    prec = args.precision or DEFAULT_PRECISION
    pipe = PhaseGenPipeline(net, N_FFT, HOP, precision=prec, per_clip=True, phase_only=True, normalize=True)
    wave = synth.synthetic_waves(1, N, SR, seed=7, device=D.dev)
    n = 50
    for _ in range(5):
        pipe(wave)
    ms_eager = D.timed(lambda: pipe(wave), n) / n
    g = pipe.capture(1, N, D.dev)
    for _ in range(5):
        g(wave)
    ms_graph = D.timed(lambda: g(wave), n) / n
    # weight bytes one forward reads: hi plane only on the two-product layers, hi + lo on the three-product ones
    params = {"d1": C * 2 * C * 32, "d2": 4 * C * C * 8, "d3": 4 * C * C * 8, "d4": 8 * C * C * 4, "u4": 8 * C * C * 5,
              "u3": 8 * C * C * 8, "u2": 8 * C * C * 8, "u1": 4 * C * C * 32}          # u1 phase-only: C of 2C outputs
    fast = set(F16MIX_FAST_LAYERS) if prec in ("f16mix", "f16mix1") else set()
    wbytes = sum(v * (2 if k in fast else 4) for k, v in params.items())
    act = 4 * N * 2 + 16 * C * T                                     # wave in/out + the few activation planes: small beside the weights
    peak = load_peaks().get("hbm_gbs") or 6650.0
    gbs = (wbytes + act) / (ms_graph / 1e3) / 1e9
    return {"metric": "single_clip_latency_ms", "workload": f"one {clip_s:.2f} s clip (N {N}), batch 1, n_fft {N_FFT}, C {C}, {prec}, device-resident",
            "ms_per_clip_eager": ms_eager, "ms_per_clip_graph": ms_graph, "audio_s_per_s_graph": clip_s / (ms_graph / 1e3),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "algorithmic_bytes": wbytes + act, "note": "weight-plane bytes of one pass + wave/activation bytes over the graph-replay time; "
                         "25 launches of 8-16 tiles each: latency-bound, not bandwidth-bound (DESIGN.md section 6)"},
            "calls_timed": n}


# ------------------------------------------------------------------------------------------ long form (config 4)
def longform_leg(args, D, net):
    """BASELINE.json config 4: a 10-minute 44.1 kHz recording (26,460,000 samples) cut into 696-frame windows with
    ~50 % overlap, windows dealt round-robin to the ranks, one all-gather of the finished windows, one stitch kernel,
    one global peak normalisation.  Strong scaling: the recording is fixed, value = 600 s / step time."""
    import torch
    from phasegen import longform, synth
    from phasegen.pipeline import PhaseGenPipeline
    minutes = args.longform_minutes
    n_total = int(minutes * 60 * SR)
    T, N, _ = workload_geometry()
    prec = args.precision or DEFAULT_PRECISION
    pipe = PhaseGenPipeline(net, N_FFT, HOP, precision=prec, per_clip=True, phase_only=True, normalize=False)
    # the same recording on every rank (seeded): 60 s of synthetic audio tiled to the full length
    base = synth.synthetic_waves(1, 60 * SR, SR, seed=11)[0]
    wave = base.repeat(-(-n_total // base.numel()))[:n_total].contiguous().to(D.dev)
    win, step, n_win = longform.window_plan(n_total, HOP, T)
    out = [None]

    def run():
        out[0] = longform.process_long(pipe, wave, frames=T, batch=CLIPS_PER_GPU + 64)
    for _ in range(2):
        run()
    ms = D.timed(run, args.steps) / args.steps
    y = out[0]
    finite = bool(torch.isfinite(y).all())
    peak = float(y.abs().max())
    # parity at full scale, measured here: (1) windows of the recording through the plain batch-1 pipeline call (the
    # demo.py:33-42 semantics) against the same windows inside this rank's long-form batch; (2) the stitch kernel on
    # all-ones windows over the full 297-window span must return exactly one everywhere (the cross-fade gains sum to one)
    wins, idx = longform.cut_windows(wave, HOP, T, D.rank, D.world)
    batch_out = pipe(wins.contiguous()).clone()
    worst = 0.0
    for j in sorted({0, len(idx) // 2, len(idx) - 1}):
        single = pipe(wins[j:j + 1].contiguous())
        worst = max(worst, float((single[0] - batch_out[j]).norm() / batch_out[j].norm()))
    ones = longform.stitch(torch.ones(n_win, win, device=D.dev), list(range(n_win)), n_win, n_total, HOP, T)
    ones_dev = float((ones - 1).abs().max())
    return {"metric": "longform_audio_seconds_per_second", "value": n_total / SR / (ms / 1e3), "unit": UNIT, "n_gpus": D.world,
            "ms_per_recording": ms, "scaling": "strong", "windows": n_win, "windows_per_rank": -(-n_win // D.world),
            "workload": f"{minutes:g}-minute recording ({n_total} samples), {n_win} windows of {T} frames, step {step} samples, "
                        f"round-robin over {D.world} rank(s), {prec}; cut + pipeline + all-gather + pg_stitch + global peak normalise",
            "finite": finite, "peak_after_normalise": peak,
            "checks": {"windows_vs_batch1_pipeline_rel_l2": worst, "stitch_of_ones_max_dev": ones_dev,
                       "pass": bool(finite and worst < 1e-4 and ones_dev < 1e-5)}}


# ------------------------------------------------------------------------------------------ GPU library arm
def run_torch_gpu(args):
    """`--impl torch_gpu`: the same 256-clip workload through stock torch on the GPU (tools/torch_baseline.py)."""
    import torch
    from phasegen import synth
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import torch_baseline
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.cuda.set_device(0)
    T, N, clip_s = workload_geometry()
    wave = synth.synthetic_waves(args.clips, N, SR, seed=100).cuda()
    res = torch_baseline.inference_baseline(wave, N_FFT, HOP, clip_s, steps=args.steps, warmup=max(args.warmup, 2))
    best = res.get("tf32", {})
    line = {"impl": "torch_gpu", "metric": METRIC, "value": best.get("value"), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 2), "ms_per_step": best.get("ms_per_step"), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "tf32 (cuDNN), fp32 elsewhere", "data": "synthetic",
            "config": {"workload": f"batched inference: {args.clips} clips x 4 s @ 44.1 kHz, n_fft {N_FFT}, hop {HOP}, T {T}, stock torch/cuDNN/cuFFT"},
            "modes": res, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DTYPE_NAMES = {"bf16x3": "bf16x3-fp32acc", "bf16": "bf16-fp32acc", "fp32_simt": "f32", "f16x3": "f16x3-fp32acc",
               "f16x2": "f16x2-fp32acc", "f16mix": "f16x3/f16x2-fp32acc (two-product fp16 on d1,u1,u2)",
               "f16mix1": "f16x3/f16x2/f16-fp32acc (two-product fp16 on d1,u2; single fp16 product = TF32 operand rounding on u1)"}
MMA_NOTES = {"bf16x3": "the fp32-class mode issues 3 bf16 MMAs per algorithmic MAC, so tensor-pipe work is 3x this figure",
             "f16x3": "3 fp16 MMAs per algorithmic MAC, so tensor-pipe work is 3x this figure",
             "f16x2": "2 fp16 MMAs per algorithmic MAC (weights rounded to fp16), tensor-pipe work is 2x this figure",
             "f16mix": "2 fp16 MMAs per algorithmic MAC on d1/u1/u2 (80 % of the MACs), 3 on the other five layers: "
                       "tensor-pipe work is 2.2x this figure",
             "f16mix1": "1 fp16 MMA per algorithmic MAC on u1 (36 % of the MACs), 2 on d1/u2 (44 %), 3 on the other five layers: "
                        "tensor-pipe work is 1.85x this figure",
             "bf16": "1 bf16 MMA per algorithmic MAC", "fp32_simt": ""}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="phasegen", choices=["phasegen", "reference", "torch_gpu"])
    ap.add_argument("--clips", type=int, default=CLIPS_PER_GPU, help="clips per GPU per step")
    ap.add_argument("--precision", default=None, choices=["bf16x3", "bf16", "fp32_simt", "f16x3", "f16mix", "f16mix1", "f16x2"],
                    help="inference default: f16mix1 (see DEFAULT_PRECISION; parity measured in every run; the all-three-product "
                         "bf16x3 and the f16mix figures are reported beside it)")
    ap.add_argument("--train-precision", default=None, choices=["bf16x3", "bf16", "fp32_simt"], help="training default: bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline leg only (no train / single / longform / library-baseline legs)")
    ap.add_argument("--e2e-chunks", type=int, default=0,
                    help="sub-batches whose copies overlap GPU work in the e2e leg (0 = wave-aligned sizes from PhaseGenPipeline.suggest_chunks)")
    ap.add_argument("--workload", default="infer", choices=["infer", "train", "single", "longform"],
                    help="infer = BASELINE config 2 (headline, default; carries the other legs as extra keys); "
                         "train = config 3; single = config 1; longform = config 4, each as its own line")
    ap.add_argument("--train-batch", type=int, default=32)
    ap.add_argument("--train-c", type=int, default=1024)
    ap.add_argument("--train-fp32", action="store_true", help="train with the fp32-class bf16x3 products instead of bf16")
    ap.add_argument("--longform-minutes", type=float, default=10.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step of the headline workload returned (rank 0) "
                         "as .npy files under DIR: the waves of evenly spaced clips, at most 64 MB")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "phasegen" or args.workload != "infer"):
        ap.error("--dump-outputs applies to the headline workload (--impl phasegen --workload infer)")
    if args.impl == "reference":
        run_reference(args)
        return
    if args.impl == "torch_gpu":
        run_torch_gpu(args)
        return

    import torch
    import model as pg_model
    from phasegen import _lib, synth
    from phasegen.pipeline import PhaseGenPipeline

    D = Dist()
    world, rank, dev = D.world, D.rank, D.dev
    if args.workload == "train":
        line = train_leg(args, D, with_library_baseline=not args.no_extras)
        if rank == 0:
            print(json.dumps(line), flush=True)
        D.close()
        return
    W = max(args.warmup, 3)
    prec = args.precision or DEFAULT_PRECISION
    T, N, clip_s = workload_geometry()
    C, B = N_FFT // 2, args.clips
    torch.manual_seed(1234)
    net = pg_model.UNetModel(C, 2 * C).to(dev)
    synth.randomize_norm_affine(net, seed=7)
    if args.workload in ("single", "longform"):
        line = single_clip_leg(args, D, net) if args.workload == "single" else longform_leg(args, D, net)
        if rank == 0:
            print(json.dumps(line), flush=True)
        D.close()
        return

    pipe = PhaseGenPipeline(net, N_FFT, HOP, precision=prec, per_clip=True, phase_only=True, normalize=True)
    host_in = synth.synthetic_waves(B, N, SR, seed=100 + rank).pin_memory()
    host_out = torch.empty(B, N, dtype=torch.float32).pin_memory()
    wave = host_in.to(dev)
    last = [None]

    def step_resident():
        last[0] = pipe(wave)

    def step_e2e_sync():
        # the public host-buffer call, one batch at a time: pinned host wave in, pinned host wave out, copies inside;
        # the call returns with its downloads ordered on the current stream
        pipe.run_host(host_in, host_out, chunks=e2e_chunks)

    # ... and as a stream of batches (the serving form, `pipelined=True`): the same copies every step, but the first
    # upload of step i+1 and the last download of step i run underneath the neighbouring step's GPU work; the result of
    # a step is awaited (event) two steps later, into alternating pinned output buffers
    host_outs = [host_out, torch.empty(B, N, dtype=torch.float32).pin_memory()]
    pend, e2e_i = [None, None], [0]

    def step_e2e():
        k = e2e_i[0] & 1
        if pend[k] is not None:
            pend[k].synchronize()                              # a consumer would read host_outs[k] here
        pend[k] = pipe.run_host(host_in, host_outs[k], chunks=stream_chunks, pipelined=True)
        e2e_i[0] += 1

    def finish_e2e():
        for ev in pend:                                        # every download of the timed steps lands inside the timed region
            if ev is not None:
                torch.cuda.current_stream().wait_event(ev)

    e2e_chunks = pipe.suggest_chunks(B, N, dev) if args.e2e_chunks == 0 else args.e2e_chunks
    # stream of batches: copies hide behind the neighbouring batches; one-wave head/tail keep the fill and drain of the timed region short
    stream_chunks = pipe.suggest_chunks(B, N, dev, stream=True) if args.e2e_chunks == 0 else args.e2e_chunks
    sampler = ClockSampler(D.local)
    if rank == 0:
        sampler.start()                                        # nvidia-smi needs ~0.1 s to deliver its first sample: start it
    for _ in range(W):                                         # before the warm-up so the timed region is covered
        step_resident()
    l0 = _lib.launches
    sampler.mark()
    ms = D.timed(step_resident, args.steps)
    launches = _lib.launches - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0])
    for _ in range(2):
        step_e2e_sync()
    ms_e2e_sync = D.timed(step_e2e_sync, args.steps)
    for _ in range(2):
        step_e2e()
    ms_e2e = D.timed(step_e2e, args.steps, finish=finish_e2e)
    torch.cuda.synchronize()
    e2e_identical = bool(torch.equal(host_outs[0], host_outs[1]))   # same input every step: both buffers hold the same waves

    audio_s = world * B * clip_s
    value = audio_s / (ms / args.steps / 1e3)
    # both host-buffer call forms are measured in every run (identical copies per step); the headline end-to-end number is the
    # faster of the two on this host (which one wins depends on the box's PCIe rate), and both are reported
    forms = {
        "stream_of_batches": {
            "value": audio_s / (ms_e2e / args.steps / 1e3), "ms_per_step": ms_e2e / args.steps, "sub_batches": stream_chunks,
            "form": "run_host(pipelined=True): every step copies its clips in from pinned host memory and its waves back out; the copies of a "
                    "step run underneath the GPU work of the neighbouring steps (two sets of staging buffers); results awaited by event, "
                    "alternating pinned output buffers"},
        "one_batch_at_a_time": {
            "value": audio_s / (ms_e2e_sync / args.steps / 1e3), "ms_per_step": ms_e2e_sync / args.steps, "sub_batches": e2e_chunks,
            "form": "run_host(): the call returns with its downloads ordered on the current stream; wave-aligned sub-batches ramp "
                    "1-2-4-..-4-2-1 waves so the copies hide inside the call"}}
    best = min(forms, key=lambda k: forms[k]["ms_per_step"])
    e2e_line = {"value": forms[best]["value"], "unit": UNIT, "h2d_bytes_per_step": B * N * 4, "d2h_bytes_per_step": B * N * 4,
                "ms_per_step": forms[best]["ms_per_step"], "sub_batches": forms[best]["sub_batches"], "form": best, "forms": forms,
                "outputs_identical_across_steps": e2e_identical, "host_binding": D.host_binding}

    # ---- roofline of the dominant kernel (conv_tc_kernel): CUDA events around every launch
    from phasegen import ops
    pending = []
    orig = ops.conv_tc

    def conv_timed(desc, *a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); orig(desc, *a, **k); e1.record()
        pending.append((e0, e1))
    # ... and of the two HBM-class kernels (stft_kernel, istft_kernel), same method
    hbm_pending = {"stft_kernel": [], "istft_kernel": []}
    orig_stft, orig_istft = ops.stft, ops.istft

    def stft_timed(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); r = orig_stft(*a, **k); e1.record()
        hbm_pending["stft_kernel"].append((e0, e1))
        return r

    def istft_timed(a, b, mode, n_fft, hop, normalize=True, check_finite=True, out=None, **kw):
        # time the ISTFT kernel alone: the peak normalisation is a separate launch (and a separate +8N-byte pass)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); w, pk = orig_istft(a, b, mode, n_fft, hop, normalize=False, check_finite=False, out=out, **kw); e1.record()
        hbm_pending["istft_kernel"].append((e0, e1))
        if normalize:
            _lib.call("pg_peak_normalize", ops._ptr(w), ops._ptr(pk), w.shape[0], w.shape[1], ops._stream())
        return w, pk
    traffic = {}
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", name)))
            break
        except OSError:
            pass
    roof = None
    peaks = load_peaks()
    if prec != "fp32_simt":
        ops.conv_tc = conv_timed
        ops.stft, ops.istft = stft_timed, istft_timed
        step_resident()                                        # one instrumented warm-up pass, not counted
        torch.cuda.synchronize()
        pending.clear()
        for v in hbm_pending.values():
            v.clear()
        for _ in range(args.steps):
            step_resident()
        torch.cuda.synchronize()
        ops.conv_tc = orig
        ops.stft, ops.istft = orig_stft, orig_istft
        tot_ms = sum(a.elapsed_time(b) for a, b in pending)
        n_launch = len(pending)
        flops_step = sum(unet_flops_per_clip(C, T, True).values()) * B
        peak = peaks.get("bf16_tflops_sustained", 1590.0 if not peaks else None) or 1590.0
        achieved = flops_step * args.steps / (tot_ms / 1e3) / 1e12
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "traffic": None, "launches": n_launch, "avg_launch_ms": tot_ms / max(n_launch, 1),
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback",
                "note": "algorithmic FLOPs (8 convs, phase-only last layer); " + MMA_NOTES[prec] +
                        "; norm statistics, normalisation, activations and the consumers' operand-plane writes run in this kernel's epilogue",
                "conv_share_of_step": (tot_ms / args.steps) / (ms / args.steps)}
        roof["traffic"] = traffic.get("conv_tc_kernel", {}).get("bytes_per_launch")
        roof["traffic_source"] = traffic.get("conv_tc_kernel", {}).get("source")
        # algorithmic bytes per clip, SURVEY.md section 8d's strict figures: STFT 4N + 4CT (the log-magnitude once: the
        # kernel writes it as the fp32 plane AND as the first convolution's operand planes, 8CT actual), ISTFT 8CT + 4N
        hbm_peak = peaks.get("hbm_gbs") or 6650.0
        alg = {"stft_kernel": B * (4 * N + 4 * C * T), "istft_kernel": B * (8 * C * T + 4 * N)}
        actual = {"stft_kernel": B * (4 * N + 8 * C * T), "istft_kernel": B * (8 * C * T + 4 * N)}
        roof_hbm = []
        for kname, evs in hbm_pending.items():
            if not evs:
                continue
            k_ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
            gbs = alg[kname] / (k_ms / 1e3) / 1e9
            roof_hbm.append({"bound": "hbm", "kernel": kname, "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                             "avg_launch_ms": k_ms, "algorithmic_bytes_per_launch": alg[kname],
                             "bytes_moved_per_launch": actual[kname], "frac_of_bytes_moved": actual[kname] / (k_ms / 1e3) / 1e9 / hbm_peak,
                             "traffic": traffic.get(kname, {}).get("bytes_per_launch"),
                             "note": "not HBM-bound: the STFT is bound by the L1TEX data pipe (shared-memory exchanges + stores, 82 % of peak), "
                                     "the ISTFT by instruction issue at low occupancy (DESIGN.md 4.2, profiles/r02_stft_pair_experiment.txt)"})
        roof["hbm_kernels"] = roof_hbm

    # ---- parity of this run, measured on clips of the timed batch
    parity = None
    if rank == 0:
        parity = measure_parity(pipe, net, wave, sorted({0, B // 2, B - 1}))

    # the all-three-product form (bf16x3: every layer at ~2^-16 per product) and the other mixed form measured beside the default
    alt = alt1 = None
    if prec in ("f16mix", "f16mix1") and not args.no_extras:
        def side_leg(p_):
            p = PhaseGenPipeline(net, N_FFT, HOP, precision=p_, per_clip=True, phase_only=True, normalize=True)
            for _ in range(2):
                p(wave)
            t = D.timed(lambda: p(wave), args.steps)
            leg = {"precision": DTYPE_NAMES[p_], "value": audio_s / (t / args.steps / 1e3), "unit": UNIT, "ms_per_step": t / args.steps}
            if rank == 0:
                par = measure_parity(p, net, wave, [B // 2])
                leg["parity"] = {k: par[k] for k in ("clips_checked", "logmag_rel_l2", "phase_rel_l2", "wave_rel_l2", "snr_db_delta", "pass")}
            return leg
        alt = side_leg("bf16x3")
        alt1 = side_leg("f16mix" if prec == "f16mix1" else "f16mix1")

    single = longf = lib = train = None
    if not args.no_extras:
        # the side legs must never cost the headline line: a leg that fails is reported as {"error": ...}
        def guarded(name, fn):
            try:
                return fn()
            except Exception as e:                               # noqa: BLE001 -- reported, not swallowed
                print(f"bench.py: leg '{name}' failed: {type(e).__name__}: {e}", file=sys.stderr, flush=True)
                return {"error": f"{type(e).__name__}: {e}"[:300]}

        def reset():
            net.__dict__["_exec"].clear(); net.__dict__["_packed"].clear()
            torch.cuda.empty_cache()
        del pipe
        reset()
        if world == 1:
            single = guarded("single_clip", lambda: single_clip_leg(args, D, net))
            reset()
        longf = guarded("longform", lambda: longform_leg(args, D, net))
        reset()
        if world == 1 and rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import torch_baseline
            lib = guarded("gpu_library_baseline", lambda: torch_baseline.inference_baseline(wave, N_FFT, HOP, clip_s, steps=3, warmup=2))
            torch.cuda.empty_cache()
        del net
        torch.cuda.empty_cache()

        def train_side():
            t = train_leg(args, D, with_library_baseline=True)
            out = {k: t[k] for k in ("metric", "value", "unit", "n_gpus", "ms_per_step", "scaling", "dtype", "config", "e2e", "gpu_launches",
                                     "roofline", "loss_trace") if k in t}
            if "gpu_library_baseline" in t:
                out["gpu_library_baseline"] = t["gpu_library_baseline"]
            return out
        train = guarded("train", train_side)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:     # reported at N = 1 only
        dt, done = cpu_reference_step(16, time_budget_s=12.0)
        cpu = {"value": clip_s * done / dt, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
               "sample": f"{done} clips of the same workload, batch-1 per clip (demo.py loop), numpy STFT/ISTFT + torch-CPU fp32 U-Net (oneDNN off)"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPE_NAMES[prec],
                "data": "synthetic",
                "config": {"workload": f"batched inference: {B} clips/GPU x 4 s @ 44.1 kHz (N {N}), n_fft {N_FFT}, hop {HOP}, "
                                       f"T {T}, U-Net C {C} (153 M params, random init), STFT->U-Net->ISTFT+peak-normalise",
                           "norm_statistics": "per clip (demo.py batch-1 semantics)", "last_layer": "phase-only",
                           "l2_policy": f"inputs larger than L2 ({B * N * 4 / 1e6:.0f} MB wave, >2 GB of activations per step)",
                           "timing": "CUDA events on the launch stream, max over ranks"},
                "e2e": e2e_line,
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "parity": parity,
                "all_three_product_form": alt, "other_mixed_form": alt1,
                "gpu_library_baseline": lib, "train": train, "single_clip": single, "longform": longf}
        print(json.dumps(line), flush=True)
    D.close()


if __name__ == "__main__":
    main()
