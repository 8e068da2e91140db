"""Cost of ragged batches (PhaseGenPipeline(..., lengths=...)) at the bench shape, in one process, one JSON line.

    python tools/ragged_bench.py [--B 256] [--steps 20] [--rounds 3] [--prec f16mix1]

(a) the fixed call against the ragged call with every length = N (N = 177,920, T = 696): the cost of the per-clip
    tables on the full-length path, next to the run-to-run spread of the fixed call.
(b) seeded lengths in [1 s, N] at 44.1 kHz: one ragged call against one fixed call per distinct frame count T_b (each
    group zero-padded to (T_b - 1)*hop, executors built and warmed before the timed window; both forms compute the
    same clips), reported as valid audio-seconds per second = sum n_b / sr / time.
Forms alternate inside every round; each time is CUDA events around `steps` back-to-back calls.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "unet-phasegen_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import model as pg_model  # noqa: E402
from phasegen import synth  # noqa: E402
from phasegen.pipeline import PhaseGenPipeline, ragged_frames  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return torch.cuda.get_device_name(), q


def timed(fn, steps):
    """ms per call over `steps` calls."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=256)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--prec", default="f16mix1")
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_bench needs a GPU")
    n_fft, hop, T, sr, B = 1024, 256, 696, 44100, a.B
    N = (T - 1) * hop
    torch.manual_seed(a.seed)
    net = pg_model.UNetModel(n_fft // 2, n_fft).cuda()
    synth.randomize_norm_affine(net, seed=a.seed + 1)
    net.max_executors = 256                                 # one per T_b group below, all kept warm
    pipe = PhaseGenPipeline(net, n_fft, hop, precision=a.prec, per_clip=True, phase_only=True)
    wave = synth.synthetic_waves(B, N, sr=sr, seed=a.seed + 2, device="cuda")
    out = torch.empty_like(wave)
    full = [N] * B

    # (a) fixed vs ragged with every length = N
    forms_a = {"fixed": lambda: pipe(wave, wave_out=out), "ragged_full": lambda: pipe(wave, wave_out=out, lengths=full)}
    for f in forms_a.values():
        for _ in range(a.warmup):
            f()
    torch.cuda.synchronize()
    ta = {k: [] for k in forms_a}
    for _ in range(a.rounds):
        for k, f in forms_a.items():
            ta[k].append(timed(f, a.steps))

    # (b) seeded lengths: one ragged call vs one fixed call per distinct T_b
    rng = np.random.default_rng(a.seed + 3)
    lengths = [int(v) for v in rng.integers(sr, N + 1, B)]
    wave_b = wave.clone()
    for i, n in enumerate(lengths):
        wave_b[i, n:] = 0.0
    groups = {}
    for i, n in enumerate(lengths):
        groups.setdefault(ragged_frames(n, hop), []).append(i)
    padded = {t: wave_b[idx, :(t - 1) * hop].contiguous() for t, idx in groups.items()}
    outs = {t: torch.empty_like(w) for t, w in padded.items()}

    def per_group():
        for t, w in padded.items():
            pipe(w, wave_out=outs[t])

    forms_b = {"ragged": lambda: pipe(wave_b, wave_out=out, lengths=lengths), "per_T_b": per_group}
    for f in forms_b.values():
        for _ in range(a.warmup):
            f()
    torch.cuda.synchronize()
    # both forms compute the same clips: largest relative L2 difference over the clips
    forms_b["ragged"]()
    per_group()
    torch.cuda.synchronize()
    diff = 0.0
    for t, idx in groups.items():
        for j, i in enumerate(idx):
            n = lengths[i]
            r, g = out[i, :n], outs[t][j, :n]
            diff = max(diff, float((r - g).norm() / g.norm()))
    tb = {k: [] for k in forms_b}
    for _ in range(a.rounds):
        for k, f in forms_b.items():
            tb[k].append(timed(f, a.steps))

    name, smi = gpu_info()
    audio_s = sum(lengths) / sr
    med = lambda v: float(np.median(v))
    line = {
        "tool": "ragged_bench", "gpu": name, "nvidia_smi_name_power_limit_max_sm_clock": smi, "precision": a.prec,
        "B": B, "n_fft": n_fft, "N": N, "steps": a.steps, "rounds": a.rounds,
        "a_fixed_ms": [round(v, 3) for v in ta["fixed"]], "a_ragged_full_ms": [round(v, 3) for v in ta["ragged_full"]],
        "a_fixed_spread_ms": round(max(ta["fixed"]) - min(ta["fixed"]), 3),
        "a_overhead_ms": round(med(ta["ragged_full"]) - med(ta["fixed"]), 3),
        "b_distinct_T_b": len(groups), "b_valid_audio_s": round(audio_s, 2),
        "b_ragged_ms": [round(v, 3) for v in tb["ragged"]], "b_per_T_b_ms": [round(v, 3) for v in tb["per_T_b"]],
        "b_ragged_audio_s_per_s": round(audio_s / (med(tb["ragged"]) / 1e3), 1),
        "b_per_T_b_audio_s_per_s": round(audio_s / (med(tb["per_T_b"]) / 1e3), 1),
        "b_max_rel_l2_ragged_vs_per_T_b": diff,
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
