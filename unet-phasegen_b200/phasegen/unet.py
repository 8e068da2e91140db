"""Executor of the U-Net forward on the phasegen kernels.

Mirrors the data flow of /root/reference/model.py (UNetModel :22-43, UNetBlock :57-113) for a
stack of D nested blocks (D = 4 in the reference), level 0 = outermost:

    down conv i   : input  = raw x (i = 0) or LeakyReLU(0.2)(h_{i-1})        model.py:90,96,103
                    h_i    = norm(z_i) for 0 < i < D-1, else z_i              (no norm outermost/innermost)
    up conv i     : input  = ReLU(z_{D-1})                      (i = D-1)     model.py:97
                             ReLU(cat[LeakyReLU(h_i), n_{i+1}])  (i < D-1)     model.py:91,104,113
                             == cat[ReLU(h_i), ReLU(n_{i+1})]   (in-place LeakyReLU quirk)
                    n_i    = norm(g_i)                                         model.py:83

Every tensor is channels-last.  The skip concat is a write at a channel offset into the up-conv's
input buffer, never a copy.  Per layer one of three forms (PG_EPI_*, include/phasegen.h):

  * fused, no norm (d1, d4): the convolution's epilogue applies the activation(s) and writes the
    consumers' 16-bit operand planes itself;
  * fused, per-clip norm (inference with per-clip statistics, whenever a clip's whole time axis fits one
    tile's 512 accumulator columns): statistics, normalisation, activation(s) and the operand-plane
    writes all happen in the epilogue -- the raw fp32 output never exists;
  * two-pass (batch statistics, training, eval-mode running statistics, the last layer): raw fp32 +
    statistics records, pg_bn_finalize, then pg_bn_act -- or, for the last layer of the fused
    pipeline, the ISTFT kernel applies (scale, shift) while it reads the raw output (`defer_last`).
"""
import torch

from . import ops
from ._lib import (PG_CONV, PG_CONV_TRANSPOSE, PG_DT_BF16, PG_DT_BF16_SPLIT, PG_DT_F16, PG_DT_F16_SPLIT, PG_DT_F32, PG_EPI_ACT,
                   PG_EPI_NORM_ACT, PG_EPI_RAW, PG_PREC_BF16, PG_PREC_BF16X3, PG_PREC_F16, PG_PREC_F16X2, PG_PREC_F16X3,
                   PG_PREC_FP32_SIMT, PRECISIONS)

BN_EPS_DEFAULT = 1e-5
# Taps that share one TMA-loaded activation strip in the tensor-core kernel (1 = no strip reuse).
# 16 with base-offset mode 0 verified on B200 against the SIMT kernel (tools/tc_probe.py,
# profiles/r01_tc_probe.log): the UMMA swizzle is a function of the absolute smem address.
DEFAULT_TAPS_PER_GROUP = 16
# precision="f16mix": layers (d<level+1> / u<level+1>) that run the two-product fp16 form.  d1, u1 and
# u2 hold 80 % of the multiply-adds of the reference U-Net (SURVEY.md section 8a); with fp16-rounded weights on
# exactly these three the predicted phase stays within ~5e-4 relative L2 of the float64 oracle
# (bound: 1e-3), measured in tests/test_gpu_unet.py.
F16MIX_FAST_LAYERS = ("d1", "u1", "u2")
# precision="f16mix1": as f16mix, plus the LAST layer (u1, 36 % of the multiply-adds) with a single fp16 product:
# both operands rounded to 11 significant bits = the operand rounding of a TF32 pass at twice its rate.  Its
# rounding error is not amplified by any later layer; measured phase error in tests/test_gpu_pipeline.py.
F16MIX1_SINGLE_LAYERS = ("u1",)
_SPLIT_PRECS = (PG_PREC_BF16X3, PG_PREC_F16X3, PG_PREC_F16X2)
_F16_PRECS = (PG_PREC_F16X3, PG_PREC_F16X2, PG_PREC_F16)
DEFAULT_BASE_OFFSET_MODE = 0


def _rows(L):
    """Allocated rows per clip: even (the stride-2 parity view reads row L when L is odd) and
    padded to 8; rows >= L stay zero forever (buffers are zero-initialised, never written).
    A ragged call (run(clip_rows=...)) also leaves rows [L_b, L) of clip b zero: every layer writes zeros there."""
    return (L + 7) // 8 * 8


def layer_lengths(levels, T):
    """Rows of every layer of a clip of T frames: [L_0 = T, L_1 .. L_D (down conv outputs), T_out (last up conv
    output)], or None when the skip concats do not line up (the reference fails in torch.cat there)."""
    Ld = [T]
    for lv in levels:
        Ld.append(lv.down.out_len(Ld[-1]))
        if Ld[-1] < 1:
            return None
    for i in range(len(levels) - 1, 0, -1):
        if levels[i].up.out_len(Ld[i + 1]) != Ld[i]:
            return None
    return Ld + [levels[0].up.out_len(Ld[1])]


def min_frames(levels, multiple=8, limit=1 << 16):
    """Smallest frame count, a multiple of `multiple`, that the U-Net accepts (24 for the reference's)."""
    for T in range(multiple, limit + 1, multiple):
        if layer_lengths(levels, T) is not None:
            return T
    raise ValueError("phasegen: no frame count up to %d fits this U-Net" % limit)


def clip_rows_table(levels, T_list):
    """Valid-row table of a ragged batch: table[j][b] = layer_lengths(levels, T_list[b])[j], j = 0 .. D+1 (the rows of
    x0, of the D down-conv outputs and of the last up-conv output).  Raises ValueError for a T the U-Net does not take."""
    cols = []
    for T in T_list:
        L = layer_lengths(levels, int(T))
        if L is None:
            raise ValueError(f"phasegen: a clip of {T} frames does not fit this U-Net (minimum {min_frames(levels)}, "
                             "and the skip connections need T % 8 == 0)")
        cols.append(L)
    return [list(r) for r in zip(*cols)]


class ConvSpec:
    def __init__(self, kind, C_in, C_out, k, stride, pad):
        self.kind, self.C_in, self.C_out, self.k, self.stride, self.pad = kind, C_in, C_out, k, stride, pad

    def out_len(self, L):
        if self.kind == PG_CONV_TRANSPOSE:
            return (L - 1) * self.stride - 2 * self.pad + self.k
        return (L + 2 * self.pad - self.k) // self.stride + 1


class LevelSpec:
    """One UNetBlock: its down conv, optional down norm, up conv, up norm."""

    def __init__(self, down, down_norm, up, up_norm=True):
        self.down, self.down_norm, self.up, self.up_norm = down, down_norm, up, up_norm


def tc_supported(levels):
    return all(l.down.C_in % 64 == 0 and l.down.C_out % 128 == 0 and l.up.C_in % 64 == 0 and l.up.C_out % 128 == 0
               for l in levels)


class _Operand:
    """Channels-last activation buffer [B][rows][ld]: fp32 (SIMT) or bf16 hi(/lo) planes."""

    def __init__(self, B, L, ld, prec, device, range_flag=None):
        self.B, self.L, self.rows, self.ld = B, L, _rows(L), ld
        self.range_flag = range_flag if prec in _F16_PRECS else None     # only fp16 planes can overflow
        if prec == PG_PREC_FP32_SIMT:
            self.dtype = PG_DT_F32
            self.hi = torch.zeros(B, self.rows, ld, device=device, dtype=torch.float32)
            self.lo = None
        elif prec == PG_PREC_F16:                      # consumed by a single-product layer: the lo plane is never read
            self.dtype = PG_DT_F16
            self.hi = torch.zeros(B, self.rows, ld, device=device, dtype=torch.float16)
            self.lo = None
        elif prec in _F16_PRECS:
            self.dtype = PG_DT_F16_SPLIT
            self.hi = torch.zeros(B, self.rows, ld, device=device, dtype=torch.float16)
            self.lo = torch.zeros_like(self.hi)
        else:
            self.dtype = PG_DT_BF16_SPLIT if prec == PG_PREC_BF16X3 else PG_DT_BF16
            self.hi = torch.zeros(B, self.rows, ld, device=device, dtype=torch.bfloat16)
            self.lo = torch.zeros_like(self.hi) if prec == PG_PREC_BF16X3 else None

    def dst(self, slope, ch_off=0):
        return ops.act_dst(self.hi, self.lo, self.rows * self.ld, self.ld, ch_off, self.dtype, slope, self.range_flag)

    def as_float(self):
        """Debug/test view: the stored value (hi + lo) as fp32 [B][L][ld]."""
        v = self.hi.float()
        if self.lo is not None:
            v = v + self.lo.float()
        return v[:, :self.L]


class UNetExecutor:
    def __init__(self, levels, B, T, device, precision="bf16x3", per_clip=False, out_channels=None,
                 taps_per_group=None, base_offset_mode=None, keep_raw=False, fast_layers=None, fuse=None,
                 use_running=False):
        """fuse: None = fuse norm / activation / operand-plane writes into the convolution epilogues wherever the
        layer allows it (tensor-core precisions, not keep_raw); False = always the two-pass form.
        use_running: normalise with the running statistics handed to run() (nn.BatchNorm eval mode)."""
        self.levels, self.B, self.T, self.device = levels, B, T, torch.device(device)
        single_layers = ()
        if precision == "f16mix1":
            precision, single_layers = "f16mix", F16MIX1_SINGLE_LAYERS
        if precision == "f16mix":
            precision, fast_layers = "f16x3", (F16MIX_FAST_LAYERS if fast_layers is None else fast_layers)
        self.prec = PRECISIONS[precision] if isinstance(precision, str) else precision
        # per-layer precision: the executor's, except that fp16 executors may run named layers two-product
        self.fast_layers = tuple(fast_layers or ()) if self.prec == PG_PREC_F16X3 else ()
        self.single_layers = tuple(single_layers) if self.prec == PG_PREC_F16X3 else ()
        if self.prec != PG_PREC_FP32_SIMT and not tc_supported(levels):
            raise RuntimeError("phasegen: tensor-core path needs C_in % 64 == 0 and C_out % 128 == 0 in every "
                               "layer; use precision='fp32_simt' for this channel count")
        self.per_clip, self.keep_raw, self.use_running = per_clip, keep_raw, bool(use_running)
        self.fuse = (self.prec != PG_PREC_FP32_SIMT and not keep_raw) if fuse is None else \
            bool(fuse and self.prec != PG_PREC_FP32_SIMT and not keep_raw)
        # sticky fp16-range flag: bit 0 set by any kernel that wrote an out-of-range value into an fp16 operand plane
        self.range_flag = torch.zeros(1, device=self.device, dtype=torch.int32)
        self.tpg = DEFAULT_TAPS_PER_GROUP if taps_per_group is None else taps_per_group
        self.bo = DEFAULT_BASE_OFFSET_MODE if base_offset_mode is None else base_offset_mode
        D = self.D = len(levels)
        dev, prec = self.device, self.prec
        # lengths: Ld[i] = rows entering down conv i; Ld[D] = innermost conv output
        self.Ld = [T]
        for lv in levels:
            self.Ld.append(lv.down.out_len(self.Ld[-1]))
            if self.Ld[-1] < 1:
                raise RuntimeError(f"phasegen: time axis too short for this U-Net (T={T})")
        for i in range(D - 1, 0, -1):
            got, want = levels[i].up.out_len(self.Ld[i + 1]), self.Ld[i]
            if got != want:
                # same failure the reference hits in torch.cat (model.py:113)
                raise RuntimeError(f"Sizes of tensors must match except in dimension 1. Expected size {want} "
                                   f"but got size {got} for the skip connection of level {i} (T={T}; "
                                   f"the reference U-Net needs T % 8 == 0 and T >= 24)")
        self.T_out = levels[0].up.out_len(self.Ld[1])
        self.C_final = levels[0].up.C_out if out_channels is None else out_channels
        G = B if per_clip else 1

        rf = self.range_flag
        self.x0 = _Operand(B, T, levels[0].down.C_in, prec, dev, rf)
        self.a, self.cat, self.z, self.g = [None] * D, [None] * D, [None] * D, [None] * D
        self.dn_desc, self.up_desc = [None] * D, [None] * D
        self.dn_mode, self.up_mode = [PG_EPI_RAW] * D, [PG_EPI_RAW] * D
        self.dn_stats, self.up_stats, self.dn_ss, self.up_ss = [None] * D, [None] * D, [None] * D, [None] * D
        self.dn_mv, self.up_mv = [None] * D, [None] * D
        for i, lv in enumerate(levels):
            Lz = self.Ld[i + 1]
            src = self.x0 if i == 0 else self.a[i - 1]
            if src.ld != lv.down.C_in:
                raise RuntimeError(f"phasegen: level {i} down conv expects {lv.down.C_in} channels, gets {src.ld}")
            self.a[i] = _Operand(B, Lz, lv.down.C_out, prec, dev, rf)   # LeakyReLU(h_i)  /  ReLU(z) innermost
            if i < D - 1:
                # [ReLU(h_i) | ReLU(n_{i+1})], read by up conv i only: planes follow that layer's precision
                cat_prec = PG_PREC_F16 if self.layer_prec("u", i) == PG_PREC_F16 else prec
                self.cat[i] = _Operand(B, Lz, lv.up.C_in, cat_prec, dev, rf)
                if lv.down.C_out + levels[i + 1].up.C_out != lv.up.C_in:
                    raise RuntimeError(f"phasegen: level {i}: concat width {lv.down.C_out}+{levels[i + 1].up.C_out} "
                                       f"!= up conv input {lv.up.C_in}")
            elif lv.up.C_in != lv.down.C_out:
                raise RuntimeError("phasegen: innermost up conv width mismatch")
            self.dn_desc[i] = ops.conv_desc(lv.down.kind, B, lv.down.C_in, lv.down.C_out, src.L, lv.down.k,
                                            lv.down.stride, lv.down.pad, src.rows, src.ld, self.layer_prec("d", i),
                                            taps_per_group=self.tpg, base_offset_mode=self.bo)
            up_src = self.a[i] if i == D - 1 else self.cat[i]
            c_out = self.C_final if i == 0 else lv.up.C_out
            self.up_desc[i] = ops.conv_desc(lv.up.kind, B, lv.up.C_in, c_out, up_src.L, lv.up.k, lv.up.stride,
                                            lv.up.pad, up_src.rows, up_src.ld, self.layer_prec("u", i),
                                            taps_per_group=self.tpg, base_offset_mode=self.bo)
            self.dn_mode[i] = self._pick_mode(self.dn_desc[i], lv.down_norm, last=False)
            self.up_mode[i] = self._pick_mode(self.up_desc[i], lv.up_norm, last=(i == 0))
            self.dn_stats[i], self.dn_ss[i], self.dn_mv[i] = self._stat_bufs(self.dn_desc[i], lv.down_norm and self.dn_mode[i] == PG_EPI_RAW, G)
            self.up_stats[i], self.up_ss[i], self.up_mv[i] = self._stat_bufs(self.up_desc[i], lv.up_norm and self.up_mode[i] == PG_EPI_RAW, G)
        # raw fp32 conv outputs (two-pass layers only): one shared scratch unless the caller wants to inspect them
        sizes = [B * self.Ld[i + 1] * levels[i].down.C_out * (self.dn_mode[i] == PG_EPI_RAW) for i in range(D)] + \
                [B * (self.T_out if i == 0 else self.Ld[i]) * self.up_desc[i].C_out * (self.up_mode[i] == PG_EPI_RAW) for i in range(D)]
        if keep_raw:
            self.z = [torch.empty(s, device=dev, dtype=torch.float32) for s in sizes[:D]]
            self.g = [torch.empty(s, device=dev, dtype=torch.float32) for s in sizes[D:]]
        else:
            scratch = torch.empty(max(max(sizes), 1), device=dev, dtype=torch.float32)
            self.z = [scratch] * D
            self.g = [scratch] * D
        self._out = None                                        # normalised last-layer output, allocated on first use
        self.weight_ready = None                                # optional callable(w): called before a kernel reads weight planes w

    @property
    def out(self):
        if self._out is None:
            self._out = torch.empty(self.B, self.T_out, self.C_final, device=self.device, dtype=torch.float32)
        return self._out

    def _pick_mode(self, desc, has_norm, last):
        """Epilogue form of a layer (module docstring).  The last layer stays two-pass: its consumer is not a
        convolution (fp32 output tensor, or the ISTFT through `defer_last`)."""
        if not self.fuse or last:
            return PG_EPI_RAW
        if not has_norm:
            return PG_EPI_ACT
        if self.per_clip and not self.use_running and ops.conv_epilogue_supported(desc, PG_EPI_NORM_ACT):
            # whole-clip tiles are OS x n_ntiles times fewer: with a small batch (the batch-1 demo.py call) they would
            # leave most of the persistent grid idle, and latency, not the normalising pass, is what counts there
            # ... and a whole clip of more than 256 accumulator columns gives up the second TMEM stage: the epilogue
            # (three passes over the accumulator) is then exposed instead of overlapped with the next tile's MMAs.
            # Measured at the BASELINE shape (tools/pipe_ab.py): +0.45 ms on d2, +0.32 ms on u3 against 0.19 / 0.14 ms
            # for their normalising pass, so a layer is fused only where its ordinary plan is single-stage anyway
            # (the two-product layers) or the whole clip still fits two stages.
            whole, split = ops.conv_plan(desc, whole_clip=1), ops.conv_plan(desc, whole_clip=0)
            if whole is not None and (whole["tiles"] >= whole["units"] or whole["tiles"] >= split["tiles"]) and \
                    whole["acc_stages"] >= split["acc_stages"]:
                return PG_EPI_NORM_ACT
        return PG_EPI_RAW

    def check_range(self):
        """Raise if any kernel of this executor wrote a value outside the fp16 range into an fp16 operand plane since
        the last check (one 4-byte device->host read).  bf16 planes have the fp32 range and never set the flag."""
        if int(self.range_flag.item()):
            self.range_flag.zero_()
            raise OverflowError("phasegen: an activation exceeded the fp16 range (|x| > 65504 or non-finite) in an fp16 "
                                "operand mode; results are invalid -- use precision='bf16x3' (bf16 planes, fp32 range)")

    def layer_prec(self, side, level):
        """Precision of the down ("d") or up ("u") convolution of a level."""
        if self.prec == PG_PREC_F16X3 and f"{side}{level + 1}" in self.single_layers:
            return PG_PREC_F16
        if self.prec == PG_PREC_F16X3 and f"{side}{level + 1}" in self.fast_layers:
            return PG_PREC_F16X2
        return self.prec

    def _stat_bufs(self, desc, has_norm, G):
        if not has_norm:
            return None, None, None
        P = ops.conv_stat_parts(desc) if self.prec != PG_PREC_FP32_SIMT else 1
        stats = torch.empty(self.B, P, desc.C_out, 4, device=self.device, dtype=torch.float32)
        ss = torch.empty(G, desc.C_out, 2, device=self.device, dtype=torch.float32)
        mv = torch.empty(G, desc.C_out, 2, device=self.device, dtype=torch.float32)
        return stats, ss, mv

    # ------------------------------------------------------------------------------ weights
    def _pack_one(self, w, kind, slice_out=None, prec=None):
        """One weight -> (hi, lo, simt).  A weight whose memory is already the packed [k][C_out][C_in]
        order (the drop-in model's) is cast elementwise; any other layout goes through the
        transposing pack kernel."""
        prec = self.prec if prec is None else prec
        tc = prec != PG_PREC_FP32_SIMT
        if not tc:
            if slice_out is not None:
                w = w[:, :slice_out]
            return ops.pack_weight(w.contiguous(), kind, want_tc=False, want_simt=True)
        plane_dtype = torch.float16 if prec in _F16_PRECS else torch.bfloat16
        want_lo = prec in (PG_PREC_BF16X3, PG_PREC_F16X3)          # the weight lo plane only feeds the third product
        pv = ops.packed_view(w, kind)
        if pv is None:
            if slice_out is not None:
                w = w[:, :slice_out]
            return ops.pack_weight(w.contiguous(), kind, want_tc=True, want_simt=False, plane_dtype=plane_dtype, want_lo=want_lo)
        if slice_out is not None:
            pv = pv[:, :slice_out].contiguous()
        hi = torch.empty(pv.shape, device=pv.device, dtype=plane_dtype)
        lo = torch.empty_like(hi) if want_lo else None
        ops.cast_split(pv, hi, lo, self.range_flag if plane_dtype == torch.float16 else None)
        return hi, lo, None

    def pack_weights(self, down_w, up_w):
        """down_w/up_w: per level, the torch-layout weights.  The final up conv is sliced to
        the first C_final output channels (phase-only inference, SURVEY section 0)."""
        self.wd, self.wu = [], []
        for i, lv in enumerate(self.levels):
            self.wd.append(self._pack_one(down_w[i], lv.down.kind, None, self.layer_prec("d", i)))
            sl = self.C_final if (i == 0 and self.C_final != lv.up.C_out) else None
            self.wu.append(self._pack_one(up_w[i], lv.up.kind, sl, self.layer_prec("u", i)))

    # ------------------------------------------------------------------------------ forward
    def _conv(self, desc, src, w, y, stats, rows=None):
        if self.weight_ready is not None:
            self.weight_ready(w)
        if rows is not None:
            ops.conv_tc(desc, src.hi, src.lo, w[0], w[1], y, stats, out_rows=rows)
            return
        if self.prec == PG_PREC_FP32_SIMT:
            ops.conv_simt(desc, src.hi, w[2], y)
            if stats is not None:
                ops.channel_stats(y, desc.B, desc.L_out, desc.C_out, desc.out_rows, desc.out_ld, stats)
        else:
            ops.conv_tc(desc, src.hi, src.lo, w[0], w[1], y, stats)

    def _finalize(self, desc, stats, ss, mv, norm, running):
        """(scale, shift) of a two-pass norm layer: from this call's statistics records, or (eval mode) from the
        running buffers."""
        gamma, beta, eps = norm
        if self.use_running:
            if running is None:
                raise RuntimeError("phasegen: executor built with use_running=True needs the running statistics")
            ops.bn_from_running(running[0], running[1], gamma, beta, eps, ss, mv)
        else:
            ops.bn_finalize(stats, desc.B, stats.shape[1], desc.C_out, self.per_clip, gamma, beta, eps, ss, mv)

    def _layer(self, mode, desc, src, w, y, stats, ss, mv, norm, running, dst0, dst1=None, rows=None):
        """One convolution + (norm) + activation fan-out, in the form chosen at construction.  rows: valid output rows
        per clip (int32 CUDA [B]) of a ragged call."""
        if mode != PG_EPI_RAW:
            if self.weight_ready is not None:
                self.weight_ready(w)
            gamma, beta, eps = norm if norm is not None else (None, None, BN_EPS_DEFAULT)
            ops.conv_tc(desc, src.hi, src.lo, w[0], w[1], None, None,
                        ops.conv_epilogue(mode, dst0, dst1, gamma, beta, eps), out_rows=rows)
            return
        self._conv(desc, src, w, y, stats, rows)
        if stats is not None:
            self._finalize(desc, stats, ss, mv, norm, running)
        ops.bn_act(y, desc.B, desc.L_out, desc.C_out, desc.out_rows, desc.out_ld,
                   ss if stats is not None else None, self.per_clip, dst0, dst1, clip_rows=rows)

    def load_input_cf(self, x):
        """x [B,C,T] fp32 (reference layout) -> the level-0 operand (one transposing kernel)."""
        B, Cn, T = x.shape
        ops.transpose(x, dst=self.x0.hi if self.x0.dtype == PG_DT_F32 else None,
                      dst_hi=None if self.x0.dtype == PG_DT_F32 else self.x0.hi, dst_lo=self.x0.lo,
                      dst_batch_stride=self.x0.rows * self.x0.ld, dst_ld=self.x0.ld, range_flag=self.x0.range_flag)

    def load_input_cl(self, x_cl):
        """x [B,T,C] fp32 channels-last -> level-0 operand (identity bn_act = cast/split)."""
        B, T, Cn = x_cl.shape
        ops.bn_act(x_cl, B, T, Cn, T, Cn, None, False, self.x0.dst(1.0))

    def run(self, dn_norm, up_norm, defer_last=False, dn_running=None, up_running=None, clip_rows=None):
        """dn_norm/up_norm: per level (gamma, beta, eps) or None.  Consumes self.x0; returns the channels-last
        output [B][T_out][C_final] (a persistent buffer of the executor).  defer_last=True skips the last layer's
        normalising pass and returns (raw output, scale_shift [G][C_final][2]) for a consumer that applies it on the
        fly (pg_istft).  dn_running/up_running: per level (running_mean, running_var) for use_running executors.
        clip_rows: ragged batch, int32 CUDA [D+2, B] = clip_rows_table(levels, T_b) with T_b <= T, x0 holding zeros in
        rows >= T_b.  Every layer then counts rows < L_b of clip b in its statistics and writes zeros into rows
        [L_b, L) of its destinations, so clip b's valid rows equal a run of that clip alone (per-clip statistics,
        tensor-core precisions).  The raw output beyond L_b is unspecified."""
        D, lv = self.D, self.levels
        if clip_rows is not None:
            if self.prec == PG_PREC_FP32_SIMT or not self.per_clip:
                raise ValueError("phasegen: ragged batches need per-clip statistics and a tensor-core precision")
            if tuple(clip_rows.shape) != (D + 2, self.B) or clip_rows.dtype != torch.int32:
                raise ValueError(f"phasegen: clip_rows must be int32 [{D + 2}, {self.B}]")
        rows = (lambda j: clip_rows[j]) if clip_rows is not None else (lambda j: None)
        run_of = lambda lst, i: lst[i] if lst is not None else None
        for i in range(D):
            src = self.x0 if i == 0 else self.a[i - 1]
            norm = dn_norm[i] if lv[i].down_norm else None
            dsts = (self.a[i].dst(0.2), self.cat[i].dst(0.0, 0)) if i < D - 1 else (self.a[i].dst(0.0), None)
            self._layer(self.dn_mode[i], self.dn_desc[i], src, self.wd[i], self.z[i], self.dn_stats[i], self.dn_ss[i],
                        self.dn_mv[i], norm, run_of(dn_running, i), *dsts, rows=rows(i + 1))
        for i in range(D - 1, 0, -1):
            src = self.a[i] if i == D - 1 else self.cat[i]
            norm = up_norm[i] if lv[i].up_norm else None
            self._layer(self.up_mode[i], self.up_desc[i], src, self.wu[i], self.g[i], self.up_stats[i], self.up_ss[i],
                        self.up_mv[i], norm, run_of(up_running, i), self.cat[i - 1].dst(0.0, lv[i - 1].down.C_out), rows=rows(i))
        # last layer: raw output + statistics, then either the normalising pass or the caller's on-the-fly affine map
        src = self.a[0] if D == 1 else self.cat[0]
        desc, y, stats = self.up_desc[0], self.g[0], self.up_stats[0]
        self._conv(desc, src, self.wu[0], y, stats, rows(D + 1))
        norm = up_norm[0] if lv[0].up_norm else None
        if norm is not None and self.C_final != lv[0].up.C_out:
            norm = (norm[0][:self.C_final] if norm[0] is not None else None,
                    norm[1][:self.C_final] if norm[1] is not None else None, norm[2])
        running = run_of(up_running, 0)
        if running is not None and self.C_final != lv[0].up.C_out:
            running = (running[0][:self.C_final], running[1][:self.C_final])
        if stats is not None:
            self._finalize(desc, stats, self.up_ss[0], self.up_mv[0], norm, running)
        if defer_last and stats is not None:
            return y[:self.B * self.T_out * self.C_final].view(self.B, self.T_out, self.C_final), self.up_ss[0]
        ops.bn_act(y, desc.B, desc.L_out, desc.C_out, desc.out_rows, desc.out_ld, self.up_ss[0] if stats is not None else None,
                   self.per_clip, ops.act_dst(self.out, None, self.T_out * self.C_final, self.C_final, 0, PG_DT_F32, 1.0),
                   clip_rows=rows(D + 1))
        return self.out
