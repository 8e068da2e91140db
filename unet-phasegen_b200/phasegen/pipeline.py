"""wave -> STFT -> U-Net -> ISTFT -> wave with every intermediate resident in HBM.

This is the path BASELINE.json's metric is quoted on: the work of the reference's
preproc_mdb.py:93 (STFT), data.py:39-47 (log-magnitude), demo.py:33-42 (per-clip U-Net
forward, polar->complex, generate_audio) for a whole batch of clips, without the
numpy/CPU round trips the reference makes at demo.py:37-40.
"""
import torch

from . import ops
from ._lib import PG_DT_F32, PG_PREC_FP32_SIMT, PG_SPEC_POLAR_LOG, PG_STFT_LOGMAG
from .unet import clip_rows_table, min_frames


def ragged_frames(n, hop):
    """Frames T_b of a clip of n samples in a ragged call: the smallest multiple of 8 with (T_b - 1)*hop >= n (the
    zero-pad-to-chunk policy of preproc_mdb.py:87-88)."""
    return (-(-n // hop) + 1 + 7) // 8 * 8


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

    def __call__(self, wave, check_finite=False, return_intermediates=False, wave_out=None, lengths=None, _precision=None):
        """wave float32 [B, N] on the GPU, N = (T-1)*hop with T % 8 == 0 -> float32 [B, N].
        check_finite=True is the finiteness check of utils.py:41 plus the fp16-range guard (one device->host sync).

        lengths (a ragged batch): B ints, clip b being wave[b, :n_b].  Its result is the standalone call on that clip
        zero-padded to (T_b - 1)*hop samples (T_b = ragged_frames(n_b)), peak normalisation included, cut to n_b
        samples; output samples [n_b, N) are 0 and wave samples >= n_b are never read.  Intermediates hold frames
        < T_b and zeros beyond.  Needs per_clip=True and a tensor-core precision; the executor is the one of the
        fixed [B, N] call.  A list of clips becomes such a call through torch.nn.utils.rnn.pad_sequence."""
        if not wave.is_cuda:
            raise RuntimeError("PhaseGenPipeline needs CUDA tensors: there is no CPU fallback")
        B, N = wave.shape
        T = self.frames(N)
        prec = _precision or self.precision
        table = self.ragged_table(B, N, lengths, prec) if lengths is not None else None
        kw = dict(self.executor_kw)
        if prec:
            kw["precision"] = prec
        ex = self.model.executor(B, T, wave.device, per_clip=self.per_clip, phase_only=self.phase_only, **kw)
        if not any(e is ex for e in self._executors):
            self._executors = (self._executors + [ex])[-8:]
        rag = {}
        if table is not None:
            table = torch.tensor(table, dtype=torch.int32).to(wave.device)   # [n_b; T_b; L_1 .. L_D; T_out]
            rag = dict(clip_rows=table[1:])
        x0 = ex.x0
        if x0.dtype != PG_DT_F32:
            # the STFT kernel writes the first convolution's 16-bit operand planes directly
            logmag, _ = ops.stft(wave, self.n_fft, self.hop, PG_STFT_LOGMAG, want_second=False,
                                 operand=(x0.hi, x0.lo, x0.rows * x0.ld),
                                 **(dict(clip_samples=table[0], clip_frames=table[1]) if rag else {}))
        else:
            logmag, _ = ops.stft(wave, self.n_fft, self.hop, PG_STFT_LOGMAG, want_second=False)
            ex.load_input_cl(logmag)
        dn, up = self.model._norm_params(wave.device)
        C = self.n_fft // 2
        ss = None
        if ex.C_final == C:
            # the last norm is applied by the ISTFT kernel while it reads the raw phase plane (no normalising pass)
            phase, ss = self.model._run(ex, dn, up, defer_last=True, **rag)
        else:
            phase = self.model._run(ex, dn, up, **rag)[:, :, :C].contiguous()      # [B, T, 2C] -> phase half
        if self._bad is None or self._bad.shape[0] < B or self._bad.device != wave.device:
            self._bad = torch.zeros(max(B, 256), device=wave.device, dtype=torch.int32)
        audio, peak = ops.istft(logmag, phase, PG_SPEC_POLAR_LOG, self.n_fft, self.hop, normalize=self.normalize,
                                check_finite=False, out=wave_out, b_scale_shift=ss, bad_out=self._bad[:B],
                                **(dict(clip_frames=table[1], clip_samples=table[0]) if rag else {}))
        if check_finite:
            try:
                ex.check_range()
            except OverflowError:
                if self.fp16_overflow == "fallback" and _precision is None:
                    return self(wave, check_finite, return_intermediates, wave_out, lengths=lengths, _precision="bf16x3")
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
        if isinstance(chunks, int):
            per = -(-B // max(1, chunks))
            sizes = [min(per, B - c0) for c0 in range(0, B, per)]
        else:
            sizes = [int(c) for c in chunks]
            if sum(sizes) != B or min(sizes) < 1:
                raise RuntimeError(f"run_host: chunk sizes {sizes} do not add up to the batch of {B}")
        cur = torch.cuda.current_stream()
        dev = cur.device
        st = getattr(self, "_host_state", None)
        key = (tuple(sizes), N, dev)
        if st is None or st["key"] != key:
            if st is not None:                              # a new batch geometry: let the old staging buffers drain before they are freed
                st["s_in"].synchronize()
                st["s_out"].synchronize()
            st = {"key": key, "s_in": torch.cuda.Stream(device=dev), "s_out": torch.cuda.Stream(device=dev), "sets": [], "calls": 0}
            self._host_state = st
        # the stream-of-batches form alternates between two sets of staging buffers, so the uploads of batch i+1 never
        # wait for batch i's GPU work (with one sub-batch per batch that is the whole difference between copy + compute
        # and max(copy, compute)); the one-batch-at-a-time form uses the first set only
        which = st["calls"] & 1 if pipelined else 0
        st["calls"] += 1 if pipelined else 0
        while len(st["sets"]) <= which:
            st["sets"].append({"d_in": [torch.empty(n, N, device=dev) for n in sizes], "d_out": [torch.empty(n, N, device=dev) for n in sizes],
                               "consumed": [None] * len(sizes), "drained": [None] * len(sizes)})
        s_in, s_out, st = st["s_in"], st["s_out"], st["sets"][which]
        if not pipelined:
            s_in.wait_stream(cur)
            s_out.wait_stream(cur)
        c0 = 0
        e_out = None
        for k, n in enumerate(sizes):
            sl = slice(c0, c0 + n)
            c0 += n
            d_in, d_out = st["d_in"][k], st["d_out"][k]
            if st["consumed"][k] is not None:
                s_in.wait_event(st["consumed"][k])          # the previous batch's sub-batch k has been read by its STFT
            with torch.cuda.stream(s_in):
                d_in.copy_(host_in[sl], non_blocking=True)
                e_in = torch.cuda.Event()
                e_in.record(s_in)
            cur.wait_event(e_in)
            if st["drained"][k] is not None:
                cur.wait_event(st["drained"][k])            # the previous batch's output k has been downloaded
            self(d_in, wave_out=d_out)
            e_done = torch.cuda.Event()
            e_done.record(cur)
            st["consumed"][k] = e_done
            s_out.wait_event(e_done)
            with torch.cuda.stream(s_out):
                host_out[sl].copy_(d_out, non_blocking=True)
                e_out = torch.cuda.Event()
                e_out.record(s_out)
            st["drained"][k] = e_out
        if pipelined:
            return e_out                                    # s_out is in order: the last download's event covers them all
        cur.wait_stream(s_out)
        return host_out


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
