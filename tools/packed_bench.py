"""Cost of packed clips (PhaseGenPipeline.packed / run_host_packed) at the bench shape, in one process, one JSON line.

    python tools/packed_bench.py [--B 256] [--steps 20] [--rounds 3] [--prec f16mix1]

256 clips with seeded lengths uniform in [1 s, N] at 44.1 kHz (N = 177,920, frames = 696).  Forms alternate inside every
round.
(a) Device-resident: the ragged call on the padded [B, N] buffer against `packed` (bitwise check of every clip); the
    STFT kernel alone, pg_stft_ragged against pg_stft_packed, with every clip offset even (float2 loads) and then every
    offset odd (scalar loads); pg_peak_normalize on [B, N] against pg_peak_normalize_packed.  CUDA events around `steps`
    back-to-back calls.
(b) From pinned host buffers: today's form (pad into a pinned [B, N] buffer on the host, one upload, the ragged call, one
    download), run_host_packed one batch at a time, and run_host_packed(pipelined=True) as a stream of batches.  Host
    clock around `steps` calls ending in a synchronise; valid audio-seconds per second = sum n_b / sr / time, and the
    bytes each form copies per call.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "unet-phasegen_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import model as pg_model  # noqa: E402
from phasegen import _lib, ops, synth  # noqa: E402
from phasegen._lib import PG_STFT_LOGMAG  # noqa: E402
from phasegen.pipeline import PhaseGenPipeline, packed_offsets  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return torch.cuda.get_device_name(), q


def timed(fn, steps):
    """ms per call over `steps` calls, CUDA events."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def host_timed(fn, steps, finish=None):
    """ms per call over `steps` calls, host clock, ending in a device synchronise."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    if finish:
        finish()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps


def rounds(forms, n_rounds, steps, warmup, timer):
    for f in forms.values():
        for _ in range(warmup):
            f()
    torch.cuda.synchronize()
    out = {k: [] for k in forms}
    for _ in range(n_rounds):
        for k, f in forms.items():
            out[k].append(timer(f, steps))
    return out


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
        raise SystemExit("packed_bench needs a GPU")
    n_fft, hop, T, sr, B = 1024, 256, 696, 44100, a.B
    N, C = (T - 1) * hop, n_fft // 2
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(a.seed)
    net = pg_model.UNetModel(C, n_fft).cuda()
    synth.randomize_norm_affine(net, seed=a.seed + 1)
    pipe = PhaseGenPipeline(net, n_fft, hop, precision=a.prec, per_clip=True, phase_only=True)
    rng = np.random.default_rng(a.seed + 3)
    lengths = [int(v) for v in rng.integers(sr, N + 1, B)]
    wave = synth.synthetic_waves(B, N, sr=sr, seed=a.seed + 2, device="cuda")
    for i, n in enumerate(lengths):
        wave[i, n:] = 0.0
    flat = torch.cat([wave[i, :n] for i, n in enumerate(lengths)])
    n_flat = flat.numel()
    out_pad, out_flat = torch.empty_like(wave), torch.empty_like(flat)
    audio_s = n_flat / sr
    med = lambda v: float(np.median(v))

    # (a) resident calls
    t_call = rounds({"ragged": lambda: pipe(wave, wave_out=out_pad, lengths=lengths),
                     "packed": lambda: pipe.packed(flat, lengths, frames=T, out=out_flat)}, a.rounds, a.steps, a.warmup, timed)
    pipe(wave, wave_out=out_pad, lengths=lengths)
    pipe.packed(flat, lengths, frames=T, out=out_flat)
    offs = packed_offsets(lengths)
    bitwise = all(torch.equal(out_flat[offs[i]:offs[i + 1]], out_pad[i, :n]) for i, n in enumerate(lengths))

    # (a) STFT kernel alone: even lengths, so every offset of `even` is even and every offset of `odd` (the same clips one
    # sample further into their buffer) is odd
    ev = [n & ~1 for n in lengths]
    tab = torch.tensor(pipe.ragged_table(B, N, ev), dtype=torch.int32, device=dev)
    off_t = torch.tensor(packed_offsets(ev), dtype=torch.int64, device=dev)
    flat_ev = torch.cat([wave[i, :n] for i, n in enumerate(ev)])
    buf = torch.empty(flat_ev.numel() + 2, device=dev)
    buf[1:1 + flat_ev.numel()] = flat_ev
    flat_odd = buf[1:1 + flat_ev.numel()]
    hi = torch.empty(B, T, C, device=dev, dtype=torch.float16)
    lo = torch.empty_like(hi)
    opd = (hi, lo, T * C)
    t_stft = rounds({
        "ragged": lambda: ops.stft(wave, n_fft, hop, PG_STFT_LOGMAG, want_second=False, operand=opd, clip_samples=tab[0], clip_frames=tab[1]),
        "packed_even": lambda: ops.stft(flat_ev, n_fft, hop, PG_STFT_LOGMAG, want_second=False, operand=opd, clip_frames=tab[1],
                                        clip_offsets=off_t, frames=T),
        "packed_odd": lambda: ops.stft(flat_odd, n_fft, hop, PG_STFT_LOGMAG, want_second=False, operand=opd, clip_frames=tab[1],
                                       clip_offsets=off_t, frames=T)}, a.rounds, 5 * a.steps, a.warmup, timed)
    ref_lm, _ = ops.stft(wave, n_fft, hop, PG_STFT_LOGMAG, want_second=False, operand=opd, clip_samples=tab[0], clip_frames=tab[1])
    odd_lm, _ = ops.stft(flat_odd, n_fft, hop, PG_STFT_LOGMAG, want_second=False, operand=opd, clip_frames=tab[1],
                         clip_offsets=off_t, frames=T)
    stft_bitwise = bool(torch.equal(ref_lm, odd_lm))

    # (a) normalise pass: in place on [B, N] against packing into the flat buffer
    peak = wave.abs().amax(1).contiguous()
    plane = out_pad.clone()
    off_full = torch.tensor(offs, dtype=torch.int64, device=dev)
    t_norm = rounds({
        "peak_normalize": lambda: _lib.call("pg_peak_normalize", ops._ptr(plane), ops._ptr(peak), B, N, ops._stream()),
        "peak_normalize_packed": lambda: ops.peak_normalize_packed(out_pad, peak, off_full, out_flat)},
        a.rounds, 5 * a.steps, a.warmup, timed)

    # (b) from pinned host buffers
    h_clips = [wave[i, :n].cpu() for i, n in enumerate(lengths)]
    h_flat = torch.cat(h_clips).pin_memory()
    h_pad_in = torch.zeros(B, N).pin_memory()
    h_pad_out = torch.empty(B, N).pin_memory()
    h_outs = [torch.empty(n_flat).pin_memory() for _ in range(2)]
    d_pad = torch.empty(B, N, device=dev)

    def padded_form():
        for i, c in enumerate(h_clips):                     # the caller's padding, on the host
            h_pad_in[i, :c.numel()].copy_(c)
        d_pad.copy_(h_pad_in, non_blocking=True)
        pipe(d_pad, wave_out=out_pad, lengths=lengths)
        h_pad_out.copy_(out_pad, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    chunks = pipe.suggest_chunks(B, N, dev)
    stream_chunks = pipe.suggest_chunks(B, N, dev, stream=True)

    def packed_form():
        pipe.run_host_packed(h_flat, lengths, h_outs[0], chunks=chunks, frames=T)
        torch.cuda.current_stream().synchronize()

    pend = [None, None]
    calls = [0]

    def stream_form():
        k = calls[0] & 1
        calls[0] += 1
        if pend[k] is not None:
            pend[k].synchronize()
        pend[k] = pipe.run_host_packed(h_flat, lengths, h_outs[k], chunks=stream_chunks, frames=T, pipelined=True)

    def stream_finish():
        for e in pend:
            if e is not None:
                e.synchronize()

    t_host = rounds({"padded_host": padded_form, "run_host_packed": packed_form},
                    a.rounds, a.steps, a.warmup, host_timed)
    t_host["run_host_packed_pipelined"] = rounds({"s": stream_form}, a.rounds, a.steps, a.warmup,
                                                 lambda f, s: host_timed(f, s, stream_finish))["s"]
    stream_finish()
    # sub-batches tile the convolutions differently from the whole batch, so the host forms are compared to the
    # resident call by their largest absolute difference (tests/test_gpu_packed.py checks them bitwise per sub-batch)
    ref = pipe.packed(flat, lengths, frames=T).cpu()       # out_flat was overwritten by the normalise timing
    host_diff = max(float((h - ref).abs().max()) for h in h_outs)

    name, smi = gpu_info()
    r = lambda v: [round(x, 3) for x in v]
    line = {
        "tool": "packed_bench", "gpu": name, "nvidia_smi_name_power_limit_max_sm_clock": smi, "precision": a.prec,
        "B": B, "n_fft": n_fft, "N": N, "frames": T, "steps": a.steps, "rounds": a.rounds,
        "valid_audio_s": round(audio_s, 2), "valid_samples": n_flat, "padded_samples": B * N,
        "a_ragged_call_ms": r(t_call["ragged"]), "a_packed_call_ms": r(t_call["packed"]),
        "a_ragged_audio_s_per_s": round(audio_s / (med(t_call["ragged"]) / 1e3), 1),
        "a_packed_audio_s_per_s": round(audio_s / (med(t_call["packed"]) / 1e3), 1),
        "a_packed_equals_ragged_bitwise": bool(bitwise),
        "a_stft_ragged_ms": r(t_stft["ragged"]), "a_stft_packed_even_ms": r(t_stft["packed_even"]),
        "a_stft_packed_odd_ms": r(t_stft["packed_odd"]), "a_stft_packed_odd_equals_ragged_bitwise": stft_bitwise,
        "a_peak_normalize_ms": r(t_norm["peak_normalize"]), "a_peak_normalize_packed_ms": r(t_norm["peak_normalize_packed"]),
        "b_chunks": chunks, "b_stream_chunks": stream_chunks,
        "b_padded_host_ms": r(t_host["padded_host"]), "b_run_host_packed_ms": r(t_host["run_host_packed"]),
        "b_run_host_packed_pipelined_ms": r(t_host["run_host_packed_pipelined"]),
        "b_padded_host_audio_s_per_s": round(audio_s / (med(t_host["padded_host"]) / 1e3), 1),
        "b_run_host_packed_audio_s_per_s": round(audio_s / (med(t_host["run_host_packed"]) / 1e3), 1),
        "b_run_host_packed_pipelined_audio_s_per_s": round(audio_s / (med(t_host["run_host_packed_pipelined"]) / 1e3), 1),
        "b_padded_host_bytes_per_call": 2 * 4 * B * N, "b_packed_bytes_per_call": 2 * 4 * n_flat,
        "b_host_max_abs_diff_vs_resident": host_diff,
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
