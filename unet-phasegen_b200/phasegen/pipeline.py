"""wave -> STFT -> U-Net -> ISTFT -> wave with every intermediate resident in HBM.

This is the path BASELINE.json's metric is quoted on: the work of the reference's
preproc_mdb.py:93 (STFT), data.py:39-47 (log-magnitude), demo.py:33-42 (per-clip U-Net
forward, polar->complex, generate_audio) for a whole batch of clips, without the
numpy/CPU round trips the reference makes at demo.py:37-40.
"""
import itertools

import torch

from . import ops
from ._lib import PG_DT_F32, PG_PREC_FP32_SIMT, PG_SPEC_POLAR_LOG, PG_STFT_LOGMAG
from .unet import clip_rows_table, min_frames


def ragged_frames(n, hop):
    """Frames T_b of a clip of n samples in a ragged call: the smallest multiple of 8 with (T_b - 1)*hop >= n (the
    zero-pad-to-chunk policy of preproc_mdb.py:87-88)."""
    return (-(-n // hop) + 1 + 7) // 8 * 8


def packed_offsets(lengths):
    """Offsets o_0 .. o_B of clips laid end to end: clip b is flat[o_b:o_(b+1)]."""
    return [0] + list(itertools.accumulate(int(v) for v in lengths))


def chunk_sizes(B, chunks, name="run_host"):
    """Sub-batch sizes of a host call: `chunks` equal ones (the last may be shorter), or an explicit list adding up to B."""
    if isinstance(chunks, int):
        per = -(-B // max(1, chunks))
        return [min(per, B - c0) for c0 in range(0, B, per)]
    sizes = [int(c) for c in chunks]
    if sum(sizes) != B or min(sizes) < 1:
        raise RuntimeError(f"{name}: chunk sizes {sizes} do not add up to the batch of {B}")
    return sizes


def packed_sub_batches(lengths, chunks):
    """Sub-batches of a packed batch for run_host_packed: per sub-batch (c0, c1, s0, s1, offsets) with clips [c0, c1),
    samples [s0, s1) of the flat buffer (one contiguous copy each way) and the offsets of its clips rebased to s0."""
    offs = packed_offsets(lengths)
    out, c0 = [], 0
    for n in chunk_sizes(len(offs) - 1, chunks, "run_host_packed"):
        c1 = c0 + n
        out.append((c0, c1, offs[c0], offs[c1], [o - offs[c0] for o in offs[c0:c1 + 1]]))
        c0 = c1
    return out


class _GraphedPipeline:
    def __init__(self, graph, static_in, static_out):
        self.graph, self.static_in, self.static_out = graph, static_in, static_out

    def __call__(self, wave):
        if tuple(wave.shape) != tuple(self.static_in.shape) or not wave.is_cuda:
            raise RuntimeError(f"graphed pipeline was captured for a CUDA tensor of shape {tuple(self.static_in.shape)}")
        self.static_in.copy_(wave, non_blocking=True)
        self.graph.replay()
        return self.static_out


class PhaseGenPipeline:
    def __init__(self, model, n_fft, hop, precision=None, per_clip=True, phase_only=True, normalize=True,
                 fp16_overflow="raise", executor_kw=None):
        """fp16_overflow: what a checked call (check_finite=True) does when an activation left the fp16 range in one
        of the fp16 operand modes: "raise" (OverflowError) or "fallback" (re-run the batch with precision="bf16x3":
        bf16 planes have the fp32 range).  Unchecked calls leave the sticky flag for `range_overflow()`."""
        ops.check_stft_geometry(n_fft, hop)
        if fp16_overflow not in ("raise", "fallback"):
            raise ValueError("fp16_overflow must be 'raise' or 'fallback'")
        self.model, self.n_fft, self.hop = model, n_fft, hop
        self.per_clip, self.phase_only, self.normalize = per_clip, phase_only, normalize
        self.precision, self.fp16_overflow = precision, fp16_overflow
        self.executor_kw = dict(executor_kw or {})     # extra UNetExecutor options (e.g. fuse=False: the two-pass norm form)
        self._executors = []
        self._bad = None
        self._planes = {}                              # packed calls' padded ISTFT planes, per (B, T, device)
        self._host_states = {}                         # run_host / run_host_packed streams and staging buffers

    def frames(self, n_samples):
        return 1 + n_samples // self.hop

    def ragged_table(self, B, N, lengths, precision=None):
        """Host int32 table [D+3][B] of a ragged call: row 0 the clip lengths n_b, rows 1 .. D+2 the valid rows of every
        layer (unet.clip_rows_table of T_b = ragged_frames(n_b)).  Raises ValueError for a call that cannot take them."""
        levels = self.model._levels()
        # resolved as in __call__ + model.executor: the call's, the pipeline's, executor_kw's, the model's
        prec = precision or self.precision or self.executor_kw.get("precision") or self.model._resolve_precision(levels)
        if prec == "fp32_simt":
            raise ValueError("lengths: ragged batches run on the tensor-core precisions only, not fp32_simt")
        if not self.per_clip:
            raise ValueError("lengths: a ragged batch needs per-clip statistics (per_clip=True); pooled statistics over "
                             "clips of different lengths have no reference meaning")
        if isinstance(lengths, torch.Tensor):
            lengths = lengths.tolist()
        n = [int(v) for v in lengths]
        if len(n) != B:
            raise ValueError(f"lengths holds {len(n)} entries for a batch of {B} clips")
        T = self.frames(N)
        if N != (T - 1) * self.hop or T % 8:
            # the kernels trust T_b <= T (rows of the executor's buffers); that holds for every n_b <= N exactly when
            # N = (T - 1)*hop with T % 8 == 0, the fixed path's own length rule
            raise ValueError(f"lengths: the [B, N] buffer must have N = (T - 1)*hop samples with T % 8 == 0 "
                             f"(got N = {N} at hop {self.hop}); pad it to such a length")
        if any(v < 0 or v > N for v in n):
            raise ValueError(f"lengths must lie in [0, {N}] (the samples of the [B, N] buffer), got {n}")
        T_min = min_frames(levels)
        T_b = [ragged_frames(v, self.hop) for v in n]
        if max(T_b) > T:                                    # cannot happen after the check above; the kernels rely on it
            raise ValueError(f"lengths: a clip needs {max(T_b)} frames, the buffer has {T}")
        short = [i for i, t in enumerate(T_b) if t < T_min]
        if short:
            raise ValueError(f"clips {short} are shorter than the {T_min} frames (at least {(T_min - 9) * self.hop + 1} "
                             f"samples at hop {self.hop}) the U-Net needs")
        return [n] + clip_rows_table(levels, T_b)

    def packed_table(self, flat, lengths, frames=None, precision=None):
        """Host tables of a packed call: (T, table, offsets).  T is the executor's frame count (`frames`, by default
        ragged_frames(max n_b)), table the ragged_table of the padded [B, (T - 1)*hop] call and offsets the B + 1 clip
        offsets in `flat`.  Raises ValueError for a call that cannot take them."""
        if flat.dim() != 1:
            raise ValueError(f"packed clips: the flat buffer must be 1-D, got shape {tuple(flat.shape)}")
        if isinstance(lengths, torch.Tensor):
            lengths = lengths.tolist()
        n = [int(v) for v in lengths]
        if not n:
            raise ValueError("packed clips: lengths is empty")
        if sum(n) != flat.numel():
            raise ValueError(f"packed clips: the lengths add up to {sum(n)} samples, the flat buffer holds {flat.numel()}")
        T_max = ragged_frames(max(n), self.hop)
        T = T_max if frames is None else int(frames)
        if T % 8 or T < T_max:
            raise ValueError(f"packed clips: frames must be a multiple of 8 and at least {T_max} (the longest clip's "
                             f"frame count), got {frames}")
        return T, self.ragged_table(len(n), (T - 1) * self.hop, n, precision), packed_offsets(n)

    def __call__(self, wave, check_finite=False, return_intermediates=False, wave_out=None, lengths=None, _precision=None):
        """wave float32 [B, N] on the GPU, N = (T-1)*hop with T % 8 == 0 -> float32 [B, N].
        check_finite=True is the finiteness check of utils.py:41 plus the fp16-range guard (one device->host sync).

        lengths (a ragged batch): B ints, clip b being wave[b, :n_b].  Its result is the standalone call on that clip
        zero-padded to (T_b - 1)*hop samples (T_b = ragged_frames(n_b)), peak normalisation included, cut to n_b
        samples; output samples [n_b, N) are 0 and wave samples >= n_b are never read.  Intermediates hold frames
        < T_b and zeros beyond.  Needs per_clip=True and a tensor-core precision; the executor is the one of the
        fixed [B, N] call.  A list of clips becomes such a call through torch.nn.utils.rnn.pad_sequence, or without
        padding through `packed`."""
        if not wave.is_cuda:
            raise RuntimeError("PhaseGenPipeline needs CUDA tensors: there is no CPU fallback")
        B, N = wave.shape
        prec = _precision or self.precision
        table = None
        if lengths is not None:                             # [n_b; T_b; L_1 .. L_D; T_out]
            table = torch.tensor(self.ragged_table(B, N, lengths, prec), dtype=torch.int32).to(wave.device)
        return self._forward(wave, B, self.frames(N), table, None, prec, check_finite, return_intermediates, wave_out,
                             _precision is None)

    def packed(self, flat, lengths, frames=None, check_finite=False, return_intermediates=False, out=None):
        """Packed clips: flat float32 1-D on the GPU holding B clips end to end (clip b = flat[o_b:o_b + n_b],
        o_b = n_0 + .. + n_(b-1), lengths = [n_0 .. n_(B-1)], sum n_b == flat.numel()) -> float32 1-D of the same
        layout.  Clip b's result, and its intermediates ([B, T, C] as in the ragged call), are bit-identical to the
        ragged call pipe(padded, lengths=lengths) on the [B, (T - 1)*hop] buffer holding clip b in row b: same
        executor, tables and kernels; only the STFT reads and the final peak-normalise pass writes the packed layout.
        frames: the executor's frame count T, by default ragged_frames(max n_b); a larger multiple of 8 keeps one
        executor for a range of batches.  out: a contiguous CUDA float32 1-D tensor of flat.numel() elements."""
        T, table, offsets = self.packed_table(flat, lengths, frames, self.precision)
        if not flat.is_cuda:
            raise RuntimeError("PhaseGenPipeline needs CUDA tensors: there is no CPU fallback")
        if out is not None and (not out.is_cuda or out.dtype != torch.float32 or out.dim() != 1 or not out.is_contiguous()
                                or out.numel() != flat.numel()):
            raise RuntimeError(f"packed: `out` must be a contiguous CUDA float32 1-D tensor of {flat.numel()} elements")
        table = torch.tensor(table, dtype=torch.int32).to(flat.device)
        offsets = torch.tensor(offsets, dtype=torch.int64).to(flat.device)
        return self._forward(flat, len(offsets) - 1, T, table, offsets, self.precision, check_finite, return_intermediates,
                             out, True)

    def _forward(self, src, B, T, table, offsets, prec, check_finite, return_intermediates, out, may_fall_back):
        """The body of a call: src [B, (T-1)*hop] (fixed or ragged: table = None or the device int32 ragged_table) or
        a packed 1-D buffer (offsets = device int64 [B+1]; its ISTFT writes a per-(B, T) scratch plane that the
        peak-normalise pass packs into `out`)."""
        kw = dict(self.executor_kw)
        if prec:
            kw["precision"] = prec
        ex = self.model.executor(B, T, src.device, per_clip=self.per_clip, phase_only=self.phase_only, **kw)
        if not any(e is ex for e in self._executors):
            self._executors = (self._executors + [ex])[-8:]
        rag = dict(clip_rows=table[1:]) if table is not None else {}
        x0 = ex.x0
        if x0.dtype != PG_DT_F32:
            # the STFT kernel writes the first convolution's 16-bit operand planes directly
            if offsets is not None:
                clips = dict(clip_frames=table[1], clip_offsets=offsets, frames=T)
            else:
                clips = dict(clip_samples=table[0], clip_frames=table[1]) if rag else {}
            logmag, _ = ops.stft(src, self.n_fft, self.hop, PG_STFT_LOGMAG, want_second=False,
                                 operand=(x0.hi, x0.lo, x0.rows * x0.ld), **clips)
        else:
            logmag, _ = ops.stft(src, self.n_fft, self.hop, PG_STFT_LOGMAG, want_second=False)
            ex.load_input_cl(logmag)
        dn, up = self.model._norm_params(src.device)
        C = self.n_fft // 2
        ss = None
        if ex.C_final == C:
            # the last norm is applied by the ISTFT kernel while it reads the raw phase plane (no normalising pass)
            phase, ss = self.model._run(ex, dn, up, defer_last=True, **rag)
        else:
            phase = self.model._run(ex, dn, up, **rag)[:, :, :C].contiguous()      # [B, T, 2C] -> phase half
        if self._bad is None or self._bad.shape[0] < B or self._bad.device != src.device:
            self._bad = torch.zeros(max(B, 256), device=src.device, dtype=torch.int32)
        packed = offsets is not None
        audio, peak = ops.istft(logmag, phase, PG_SPEC_POLAR_LOG, self.n_fft, self.hop, normalize=self.normalize and not packed,
                                check_finite=False, out=self._packed_plane(B, T, src.device) if packed else out,
                                b_scale_shift=ss, bad_out=self._bad[:B],
                                **(dict(clip_frames=table[1], clip_samples=table[0]) if rag else {}))
        if packed:
            # the normalise pass packs the padded plane (a copy when normalize=False): no extra pass over the audio
            audio = ops.peak_normalize_packed(audio, peak if self.normalize else None, offsets,
                                              out if out is not None else torch.empty(src.numel(), device=src.device))
        if check_finite:
            try:
                ex.check_range()
            except OverflowError:
                if self.fp16_overflow == "fallback" and may_fall_back:
                    return self._forward(src, B, T, table, offsets, "bf16x3", check_finite, return_intermediates, out, False)
                raise
            if bool(self._bad[:B].any().item()):
                raise ValueError("Audio buffer is not finite everywhere")
        if return_intermediates:
            if ss is not None:                                  # the normalised phase, materialised for inspection only
                phase_n = torch.empty_like(phase)
                ops.bn_act(phase, B, T, C, T, C, ss, self.per_clip, ops.act_dst(phase_n, None, T * C, C, 0, PG_DT_F32, 1.0),
                           clip_rows=table[-1] if rag else None)
                phase = phase_n
            return audio, logmag, phase
        return audio

    def _packed_plane(self, B, T, device):
        """The padded [B, (T - 1)*hop] ISTFT output of packed calls: scratch, one per (B, T, device)."""
        planes = self._planes
        key = (B, T, device)
        if key not in planes:
            if len(planes) >= 8:
                planes.clear()
            planes[key] = torch.empty(B, (T - 1) * self.hop, device=device)
        return planes[key]

    def range_overflow(self):
        """Sticky fp16-range flags of every executor this pipeline has used, read and cleared (one small device->host
        read per executor): True means some activation left the fp16 range since the last call."""
        hit = False
        for ex in self._executors:
            if int(ex.range_flag.item()):
                ex.range_flag.zero_()
                hit = True
        return hit

    def nonfinite_clips(self, B):
        """Per-clip non-finite flags of the LAST call (utils.py:41), as a host list."""
        return [] if self._bad is None else [i for i, v in enumerate(self._bad[:B].tolist()) if v]

    def capture(self, B, n_samples, device=None, warmup=2):
        """CUDA-graph form of the pipeline for one fixed shape: the ~25 launches of a call are recorded once and
        replayed with a single `cudaGraphLaunch`, which removes the per-launch host cost (0.8 ms of Python/ctypes
        per call -- comparable to the 1.3 ms of GPU time of a single 4 s clip).  Returns a callable
        ``g(wave) -> audio``: `wave` is copied into the graph's static input buffer, the result is the graph's
        static output buffer (valid until the next call; clone it to keep it).  Weights are read from the
        executor's packed planes at replay time: call ``capture`` again after changing the model's weights."""
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        static_in = torch.zeros(B, n_samples, device=dev, dtype=torch.float32)
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):                   # warm-up off the capture: executors, packed weights, smem opt-ins
            for _ in range(max(1, warmup)):
                self(static_in)
        cur.wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_out = self(static_in)
        return _GraphedPipeline(graph, static_in, static_out)

    def suggest_chunks(self, B, n_samples, device, max_waves=6, stream=False):
        """Sub-batch sizes for run_host.  Every size fills whole waves of the persistent grid in the heaviest convolution
        (a sub-batch that spills a few tiles into an extra wave pays for the whole wave), and the sizes RAMP: 1, 2, 4
        waves at the head, `max_waves` in the middle, 4, 2, 1 at the tail.  The upload of sub-batch j+1 has to land while
        sub-batch j computes, and the download of sub-batch j-1 has to drain while j computes: with a one-wave head
        followed directly by a six-wave sub-batch the second upload needed ~49 GB/s of PCIe to keep the GPU busy
        (78 MB during 1.6 ms); the ramp needs a third of that, and the exposed first upload / last download stay one wave
        long.  From the tiling plan of the outermost up convolution."""
        import ctypes
        from . import _lib
        T = self.frames(n_samples)
        kw = dict(self.executor_kw)
        if self.precision:
            kw["precision"] = self.precision
        ex = self.model.executor(B, T, device, per_clip=self.per_clip, phase_only=self.phase_only, **kw)
        out = (ctypes.c_int * 16)()
        if ex.prec == _lib.PG_PREC_FP32_SIMT or _lib.load().pg_conv_tc_plan(ctypes.byref(ex.up_desc[0]), out, 16) != 0:
            return [B]
        n_ntiles, nb, pair, n_cotiles, OS = out[1], out[2], out[4], out[9], out[10]
        slabs = (n_cotiles // 2 if pair else n_cotiles) * OS * n_ntiles
        units = 74 if pair else 148
        cap = lambda waves: max(nb, nb * ((waves * units) // slabs))
        if stream:
            # stream of batches (run_host(pipelined=True)): copies hide behind the neighbouring batches whatever the sizes, so
            # the middle is ONE sub-batch (no tiling loss); the one-wave head and tail only keep the pipeline's fill (first
            # upload) and drain (last download), which a benchmark's timed region -- or a short burst of batches -- pays in full
            return [cap(1), B - 2 * cap(1), cap(1)] if B > 4 * cap(1) else [B]
        return ramp_sizes(B, cap, nb, max_waves)

    def run_host(self, host_in, host_out, chunks=4, pipelined=False):
        """End-to-end call on HOST buffers (pinned float32 [B, N] in and out): the batch is cut into
        sub-batches (`chunks`: how many equal ones, or an explicit list of sizes, e.g. from suggest_chunks)
        whose host->device copy, GPU work and device->host copy overlap on three streams.  Every sub-batch has its
        own persistent device staging buffers (in and out: 2 x 4 B per sample of the batch in total, allocated once per
        batch geometry), so the upload stream never waits for a free slot: it runs ahead of the GPU work by as much as
        the PCIe rate allows.  Returns when every download has been ordered on the current stream (synchronise it
        before reading host_out).

        pipelined=True is the serving form for a stream of batches: the call does not order its copies against the
        current stream at entry or exit and alternates between two sets of staging buffers, so the uploads of batch i+1
        run underneath the GPU work of batch i and the downloads of batch i underneath batch i+1 (each staging buffer
        is guarded by its own events: an upload waits until the batch two calls back has been read from it, a sub-batch
        waits until its previous output has drained).  Throughput is then max(copies, GPU work) for any `chunks`,
        including a single sub-batch (`chunks=1`: no sub-batch tiling loss at all); sub-batches only shorten the latency
        of one batch.
        The caller promises that `host_in` is ready when the call is made, gives consecutive calls different
        `host_out` buffers, and waits on the returned event (``ev.synchronize()`` or ``stream.wait_event(ev)``)
        before reading `host_out`."""
        if host_in.is_cuda or host_out.is_cuda:
            raise RuntimeError("run_host takes host tensors; call the pipeline directly for device tensors")
        B, N = host_in.shape
        sizes = chunk_sizes(B, chunks)
        starts = list(itertools.accumulate([0] + sizes))
        dev = torch.cuda.current_stream().device
        e_out = self._host_loop(
            ("rows", tuple(sizes), N, dev), sizes, pipelined,
            stage=lambda n: (torch.empty(n, N, device=dev), torch.empty(n, N, device=dev)),
            upload=lambda k, d_in: d_in.copy_(host_in[starts[k]:starts[k + 1]], non_blocking=True),
            compute=lambda k, d_in, d_out, tab: self(d_in, wave_out=d_out),
            download=lambda k, d_out: host_out[starts[k]:starts[k + 1]].copy_(d_out, non_blocking=True))
        return e_out if pipelined else host_out

    def run_host_packed(self, host_in, lengths, host_out, chunks=4, frames=None, pipelined=False):
        """`packed` on HOST buffers: pinned float32 1-D in and out, clips end to end as in `packed`, with the contract
        of run_host (sub-batches whose copies overlap the GPU work; pipelined=True returns the event of the last
        download).  Sub-batch k holds clips [c0, c0 + n) and copies samples [o_c0, o_(c0+n)) in and out, one
        contiguous copy each way, so no padding crosses PCIe.  Every sub-batch runs at the same frame count T
        (`frames`, by default that of the longest clip of the batch); its staging buffers hold n*(T - 1)*hop samples
        and are allocated once per (sub-batch sizes, T, device), so a stream of batches with different lengths and
        the same `frames` reuses them.  The per-clip tables of all sub-batches are uploaded in one copy from a pinned
        buffer before the first sub-batch's samples.  suggest_chunks(B, (T - 1)*hop, device[, stream=True]) gives
        sub-batch sizes that fill whole waves of the convolution grid.  Each clip's result is bit-identical to
        `packed` on its sub-batch with the same `frames`."""
        if host_in.is_cuda or host_out.is_cuda:
            raise RuntimeError("run_host_packed takes host tensors; call `packed` for device tensors")
        T, table, _ = self.packed_table(host_in, lengths, frames, self.precision)
        if host_out.dim() != 1 or host_out.numel() != host_in.numel():
            raise RuntimeError(f"run_host_packed: host_out must be 1-D with {host_in.numel()} elements")
        subs = packed_sub_batches(table[0], chunks)
        sizes = [c1 - c0 for c0, c1, _, _, _ in subs]
        R = len(table)
        # one host buffer for every sub-batch's tables: the int64 rebased offsets of all sub-batches, then their int32
        # [R, n] ragged tables (every part a multiple of 8 bytes long when it is int64, so each view stays aligned)
        parts = [torch.tensor(o, dtype=torch.int64).view(torch.uint8) for _, _, _, _, o in subs]
        parts += [torch.tensor([row[c0:c1] for row in table], dtype=torch.int32).view(-1).view(torch.uint8)
                  for c0, c1, _, _, _ in subs]
        at = list(itertools.accumulate([0] + [p.numel() for p in parts]))
        tables = torch.cat(parts)
        K = len(subs)
        span = (T - 1) * self.hop
        dev = torch.cuda.current_stream().device

        def compute(k, d_in, d_out, tab):
            c0, c1, s0, s1, _ = subs[k]
            offs = tab[at[k]:at[k + 1]].view(torch.int64)
            rows = tab[at[K + k]:at[K + k + 1]].view(torch.int32).view(R, c1 - c0)
            self._forward(d_in[:s1 - s0], c1 - c0, T, rows, offs, self.precision, False, False, d_out[:s1 - s0], False)

        e_out = self._host_loop(
            ("packed", tuple(sizes), T, dev, tables.numel()), sizes, pipelined,
            stage=lambda n: (torch.empty(n * span, device=dev), torch.empty(n * span, device=dev)),
            upload=lambda k, d_in: d_in[:subs[k][3] - subs[k][2]].copy_(host_in[subs[k][2]:subs[k][3]], non_blocking=True),
            compute=compute,
            download=lambda k, d_out: host_out[subs[k][2]:subs[k][3]].copy_(d_out[:subs[k][3] - subs[k][2]], non_blocking=True),
            tables=tables)
        return e_out if pipelined else host_out

    def _host_loop(self, key, sizes, pipelined, stage, upload, compute, download, tables=None):
        """The stream / event / staging loop of run_host and run_host_packed.  key[0] names the form; a new key
        replaces that form's streams and buffers.  stage(n) -> (d_in, d_out), the device staging buffers of a sub-batch
        of n clips (allocated once per key and staging set); upload(k, d_in) and download(k, d_out) enqueue the copies
        of sub-batch k (on the upload / download stream), compute(k, d_in, d_out, tab) its GPU work (on the current
        stream).  tables (CPU uint8, the same size for every call of a key): copied into the set's pinned buffer and
        uploaded in one copy ahead of the first sub-batch; compute receives the device copy.  Returns the event of the
        last download (pipelined) or None after ordering the downloads on the current stream."""
        cur = torch.cuda.current_stream()
        dev = cur.device
        st = self._host_states.get(key[0])
        if st is None or st["key"] != key:
            if st is not None:                              # a new batch geometry: let the old staging buffers drain before they are freed
                st["s_in"].synchronize()
                st["s_out"].synchronize()
            st = {"key": key, "s_in": torch.cuda.Stream(device=dev), "s_out": torch.cuda.Stream(device=dev), "sets": [], "calls": 0}
            self._host_states[key[0]] = st
        # the stream-of-batches form alternates between two sets of staging buffers, so the uploads of batch i+1 never
        # wait for batch i's GPU work (with one sub-batch per batch that is the whole difference between copy + compute
        # and max(copy, compute)); the one-batch-at-a-time form uses the first set only
        which = st["calls"] & 1 if pipelined else 0
        st["calls"] += 1 if pipelined else 0
        while len(st["sets"]) <= which:
            bufs = [stage(n) for n in sizes]
            st["sets"].append({"d_in": [b[0] for b in bufs], "d_out": [b[1] for b in bufs],
                               "consumed": [None] * len(sizes), "drained": [None] * len(sizes),
                               "tab_host": None, "tab_dev": None, "tab_sent": None})
        s_in, s_out, st = st["s_in"], st["s_out"], st["sets"][which]
        if not pipelined:
            s_in.wait_stream(cur)
            s_out.wait_stream(cur)
        tab = None
        if tables is not None:
            if st["tab_host"] is None:
                st["tab_host"] = torch.empty_like(tables).pin_memory()
                st["tab_dev"] = torch.empty_like(tables, device=dev)
            elif st["tab_sent"] is not None:
                st["tab_sent"].synchronize()                # the last upload from the pinned buffer has read it
            st["tab_host"].copy_(tables)
            if st["consumed"][-1] is not None:
                s_in.wait_event(st["consumed"][-1])         # the previous batch on this set has run (and read the tables)
            with torch.cuda.stream(s_in):
                st["tab_dev"].copy_(st["tab_host"], non_blocking=True)
                st["tab_sent"] = torch.cuda.Event()
                st["tab_sent"].record(s_in)
            tab = st["tab_dev"]
        e_out = None
        for k in range(len(sizes)):
            d_in, d_out = st["d_in"][k], st["d_out"][k]
            if st["consumed"][k] is not None:
                s_in.wait_event(st["consumed"][k])          # the previous batch's sub-batch k has been read by its STFT
            with torch.cuda.stream(s_in):
                upload(k, d_in)
                e_in = torch.cuda.Event()
                e_in.record(s_in)
            cur.wait_event(e_in)
            if st["drained"][k] is not None:
                cur.wait_event(st["drained"][k])            # the previous batch's output k has been downloaded
            compute(k, d_in, d_out, tab)
            e_done = torch.cuda.Event()
            e_done.record(cur)
            st["consumed"][k] = e_done
            s_out.wait_event(e_done)
            with torch.cuda.stream(s_out):
                download(k, d_out)
                e_out = torch.cuda.Event()
                e_out.record(s_out)
            st["drained"][k] = e_out
        if pipelined:
            return e_out                                    # s_out is in order: the last download's event covers them all
        cur.wait_stream(s_out)
        return None


def ramp_sizes(B, cap, nb, max_waves=6):
    """Sub-batch sizes [cap(1), cap(2), cap(4), cap(max_waves) ..., cap(4), cap(2), cap(1)] adding up to B (cap(w) = clips whose
    tiles fill at most w waves; sizes are multiples of nb except possibly one).  Short batches drop the outer steps."""
    for steps in ((1, 2, 4), (1, 2), (1,)):
        head = [cap(w) for w in steps]
        rest = B - 2 * sum(head)
        if rest >= nb:
            mid, sizes = cap(max_waves), []
            while rest > 0:
                sizes.append(min(mid, rest))
                rest -= sizes[-1]
            if len(sizes) > 1 and sizes[-1] < sizes[-2]:    # split the remainder evenly over the last two middles
                tot = sizes[-1] + sizes[-2]
                a = (tot // 2 + nb - 1) // nb * nb
                sizes[-2], sizes[-1] = a, tot - a
            return head + sizes + head[::-1]
    return [B]
