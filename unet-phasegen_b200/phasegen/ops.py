"""Tensor-level wrappers over the phasegen C ABI (torch is used for device memory and
streams only; every arithmetic step below is a kernel of libphasegen.so)."""
import ctypes as C
import math

import torch

from . import _lib
from ._lib import (ActDst, ConvDesc, ConvEpilogue, PG_EPI_ACT, PG_EPI_NORM_ACT, PG_EPI_RAW, PG_CONV, PG_CONV_TRANSPOSE, PG_DT_BF16, PG_DT_BF16_SPLIT, PG_DT_F16,
                   PG_DT_F16_SPLIT, PG_DT_F32, PG_DT_NONE, PG_FMT_BF16, PG_FMT_F16, PG_PREC_BF16, PG_PREC_BF16X3,
                   PG_PREC_F16X2, PG_PREC_F16X3, PG_PREC_FP32_SIMT, PG_SPEC_CARTESIAN, PG_SPEC_POLAR_LOG,
                   PG_SPEC_POLAR_MAG, PG_STFT_LOGMAG, PG_STFT_REIM)

SUPPORTED_N_FFT = (256, 512, 1024, 2048)


def _stream(t=None):
    """The current stream of the device `t` lives on (of the current device when no tensor is given)."""
    dev = t.device if isinstance(t, torch.Tensor) and t.is_cuda else None
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _fmt(t):
    """16-bit operand format of a plane tensor (None -> bf16)."""
    if t is None or t.dtype == torch.bfloat16:
        return PG_FMT_BF16
    if t.dtype == torch.float16:
        return PG_FMT_F16
    raise RuntimeError(f"phasegen: operand planes must be bfloat16 or float16, got {t.dtype}")


def _need_cuda(t, name, dtype=torch.float32):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"phasegen: `{name}` must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise RuntimeError(f"phasegen: `{name}` must be {dtype}, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        # kernels are launched on the CURRENT device's stream: a tensor elsewhere would be read from the wrong device
        raise RuntimeError(f"phasegen: `{name}` lives on {t.device} but the current device is cuda:{torch.cuda.current_device()}; "
                           "wrap the call in `with torch.cuda.device(tensor.device):`")
    _lib.require_device(t.device.index)
    return t.contiguous()


_twiddles = {}


def twiddle(n_fft, device):
    """float2[n_fft] table exp(-2 pi i m / n_fft), computed in float64 on the host once."""
    key = (n_fft, str(device))
    if key not in _twiddles:
        m = torch.arange(n_fft, dtype=torch.float64)
        ang = -2.0 * math.pi * m / n_fft
        _twiddles[key] = torch.stack([torch.cos(ang), torch.sin(ang)], 1).float().contiguous().to(device)
    return _twiddles[key]


def check_stft_geometry(n_fft, hop):
    if n_fft not in SUPPORTED_N_FFT or hop * 4 != n_fft:
        raise RuntimeError(f"phasegen: n_fft must be one of {SUPPORTED_N_FFT} with hop = n_fft/4 "
                           f"(got n_fft={n_fft}, hop={hop})")


def _lengths(t, B, name, dtype=torch.int32):
    """A per-clip table argument: a contiguous int32 (int64 for offsets) CUDA tensor of B entries."""
    t = _need_cuda(t, name, dtype)
    if t.numel() != B:
        raise RuntimeError(f"phasegen: `{name}` must hold one entry per clip ({B}), got {t.numel()}")
    return t


def stft(wave, n_fft, hop, mode=PG_STFT_LOGMAG, want_second=True, operand=None, clip_samples=None, clip_frames=None,
         clip_offsets=None, frames=None):
    """wave [B,N] -> (a, b) fp32 [B,T,n_fft/2] frame-major, DC bin dropped.
    mode LOGMAG: a = log1p|X|, b = angle X;  REIM: a = Re X, b = Im X.
    operand = (hi, lo, batch_stride): also write `a` as bf16 planes (first-conv operand).
    clip_samples / clip_frames (ragged batch, LOGMAG only): int32 CUDA [B], n_b and T_b of each clip (pg_stft_ragged):
    clip b is its first n_b samples zero-padded to (T_b - 1)*hop, frames >= T_b are 0.
    clip_offsets (packed clips, LOGMAG only, with clip_frames and `frames` = T): int64 CUDA [B+1]; wave is 1-D and clip b
    is wave[o_b:o_(b+1)], otherwise as the ragged batch (pg_stft_packed)."""
    check_stft_geometry(n_fft, hop)
    wave = _need_cuda(wave, "wave")
    if clip_offsets is not None:
        if wave.dim() != 1 or frames is None or clip_frames is None:
            raise RuntimeError("phasegen.stft: packed clips need a 1-D wave, clip_frames and frames")
        B, T, Cb = clip_offsets.numel() - 1, int(frames), n_fft // 2
        a = torch.empty(B, T, Cb, device=wave.device, dtype=torch.float32)
        b = torch.empty_like(a) if want_second else None
        hi, lo, bs = operand if operand is not None else (None, None, 0)
        _lib.call("pg_stft_packed", _ptr(wave), wave.numel(), _ptr(_lengths(clip_offsets, B + 1, "clip_offsets", torch.int64)),
                  B, T, n_fft, hop, _ptr(twiddle(n_fft, wave.device)), mode, _ptr(a), _ptr(b), _ptr(hi), _ptr(lo), bs,
                  _fmt(hi), _ptr(_lengths(clip_frames, B, "clip_frames")), _stream())
        return a, b
    if wave.dim() != 2:
        raise RuntimeError("phasegen.stft: wave must be [B, N]")
    B, N = wave.shape
    T = 1 + N // hop
    Cb = n_fft // 2
    a = torch.empty(B, T, Cb, device=wave.device, dtype=torch.float32)
    b = torch.empty_like(a) if want_second else None
    hi, lo, bs = operand if operand is not None else (None, None, 0)
    if clip_samples is not None or clip_frames is not None:
        _lib.call("pg_stft_ragged", _ptr(wave), B, N, n_fft, hop, _ptr(twiddle(n_fft, wave.device)), mode,
                  _ptr(a), _ptr(b), _ptr(hi), _ptr(lo), bs, _fmt(hi), _ptr(_lengths(clip_samples, B, "clip_samples")),
                  _ptr(_lengths(clip_frames, B, "clip_frames")), _stream())
        return a, b
    _lib.call("pg_stft", _ptr(wave), B, N, n_fft, hop, _ptr(twiddle(n_fft, wave.device)), mode,
              _ptr(a), _ptr(b), _ptr(hi), _ptr(lo), bs, _fmt(hi), _stream())
    return a, b


def stft_project(wave, mag, n_fft, hop, out=None):
    """One Griffin-Lim projection: STFT of wave [B,N], phase kept, magnitude replaced by mag [B,T,C]
    -> (re, im) fp32 [B,T,C] for istft(..., PG_SPEC_CARTESIAN).  `out` = (re, im) buffers to reuse."""
    check_stft_geometry(n_fft, hop)
    wave = _need_cuda(wave, "wave")
    mag = _need_cuda(mag, "mag")
    B, N = wave.shape
    T = 1 + N // hop
    if tuple(mag.shape) != (B, T, n_fft // 2):
        raise RuntimeError(f"phasegen.stft_project: mag must be [{B}, {T}, {n_fft // 2}], got {tuple(mag.shape)}")
    re, im = out if out is not None else (torch.empty_like(mag), torch.empty_like(mag))
    _lib.call("pg_stft_project", _ptr(wave), B, N, n_fft, hop, _ptr(twiddle(n_fft, wave.device)), _ptr(mag),
              _ptr(re), _ptr(im), _stream())
    return re, im


def stft_pairs(wave, n_fft, hop, mean=0.0, std=1.0):
    """wave [B,N] -> (log1p|X'|, angle X') fp32 [B,T,C] with X' = (X - mean(1+j)) / std: the STFT of
    preproc_mdb.py:93-96, the dataset standardisation of :182 and data.py:39-47 in one kernel."""
    check_stft_geometry(n_fft, hop)
    wave = _need_cuda(wave, "wave")
    B, N = wave.shape
    T = 1 + N // hop
    lm = torch.empty(B, T, n_fft // 2, device=wave.device, dtype=torch.float32)
    ph = torch.empty_like(lm)
    _lib.call("pg_stft_pairs", _ptr(wave), B, N, n_fft, hop, _ptr(twiddle(n_fft, wave.device)), float(mean), float(std),
              _ptr(lm), _ptr(ph), _stream())
    return lm, ph


def istft(a, b, mode, n_fft, hop, normalize=True, check_finite=True, out=None, b_scale_shift=None, bad_out=None,
          clip_frames=None, clip_samples=None):
    """(a, b) fp32 [B,T,n_fft/2] frame-major -> wave [B,(T-1)*hop]; optional peak normalisation
    (utils.py:42) and finiteness check (utils.py:41; costs one device->host sync).
    b_scale_shift: float2 per bin, [B, C, 2] (per clip) or [1, C, 2] / [C, 2]: b is read as b*scale + shift (the final
    norm of the U-Net applied on the fly).  bad_out: int32 [B] buffer that receives the per-clip non-finite flags.
    clip_frames / clip_samples (ragged batch): int32 CUDA [B], T_b and n_b of each clip (pg_istft_ragged): clip b is
    reconstructed from its first T_b frames, its peak and flags cover (T_b - 1)*hop samples, samples >= n_b are 0."""
    check_stft_geometry(n_fft, hop)
    a = _need_cuda(a, "a")
    b = _need_cuda(b, "b") if b is not None else None
    B, T, Cb = a.shape
    if Cb != n_fft // 2 or (b is not None and b.shape != a.shape):
        raise RuntimeError("phasegen.istft: inputs must be [B, T, n_fft/2] and of equal shape")
    n = (T - 1) * hop
    if out is not None and (tuple(out.shape) != (B, n) or out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous()):
        raise RuntimeError(f"phasegen.istft: `out` must be a contiguous CUDA float32 [{B}, {n}] tensor")
    wave = out if out is not None else torch.empty(B, n, device=a.device, dtype=torch.float32)
    peak = torch.empty(B, device=a.device, dtype=torch.float32)
    bad = bad_out if bad_out is not None else torch.empty(B, device=a.device, dtype=torch.int32)
    per_clip = 0
    if b_scale_shift is not None:
        b_scale_shift = _need_cuda(b_scale_shift, "b_scale_shift")
        if b_scale_shift.numel() not in (2 * Cb, 2 * Cb * B):
            raise RuntimeError("phasegen.istft: b_scale_shift must hold (scale, shift) per bin, for all clips or per clip")
        per_clip = int(b_scale_shift.numel() == 2 * Cb * B and B > 1)
    if clip_frames is not None or clip_samples is not None:
        _lib.call("pg_istft_ragged", _ptr(a), _ptr(b), mode, B, T, n_fft, hop, _ptr(twiddle(n_fft, a.device)),
                  _ptr(wave), _ptr(peak), _ptr(bad), _ptr(b_scale_shift), per_clip,
                  _ptr(_lengths(clip_frames, B, "clip_frames")), _ptr(_lengths(clip_samples, B, "clip_samples")), _stream())
    else:
        _lib.call("pg_istft", _ptr(a), _ptr(b), mode, B, T, n_fft, hop, _ptr(twiddle(n_fft, a.device)),
                  _ptr(wave), _ptr(peak), _ptr(bad), _ptr(b_scale_shift), per_clip, _stream())
    if normalize:
        _lib.call("pg_peak_normalize", _ptr(wave), _ptr(peak), B, n, _stream())
    if check_finite and bool(bad.any().item()):
        raise ValueError("Audio buffer is not finite everywhere")
    return wave, peak


def peak_normalize_packed(src, peak, clip_offsets, out):
    """Pack the rows of src [B, n] (an ISTFT output) into out [sum n_b] (pg_peak_normalize_packed):
    out[o_b + i] = src[b, i] / peak[b] for i < n_b = o_(b+1) - o_b, the pg_peak_normalize rule; a copy when peak is None.
    clip_offsets: int64 CUDA [B+1]."""
    src = _need_cuda(src, "src")
    if src.dim() != 2:
        raise RuntimeError("phasegen.peak_normalize_packed: src must be [B, n]")
    B = src.shape[0]
    peak = _lengths(peak, B, "peak", torch.float32) if peak is not None else None
    offs = _lengths(clip_offsets, B + 1, "clip_offsets", torch.int64)
    if not (isinstance(out, torch.Tensor) and out.dim() == 1 and out.is_contiguous()):
        raise RuntimeError("phasegen.peak_normalize_packed: `out` must be a contiguous 1-D CUDA float32 tensor")
    _need_cuda(out, "out")
    _lib.call("pg_peak_normalize_packed", _ptr(src), B, src.shape[1], _ptr(peak), _ptr(offs), _ptr(out), out.numel(), _stream())
    return out


def transpose(src, dst=None, dst_hi=None, dst_lo=None, dst_batch_stride=None, dst_ld=None, range_flag=None):
    """[B,R,S] fp32 -> [B,S,R] (fp32 and/or bf16 hi/lo planes with the given pitch)."""
    src = _need_cuda(src, "src")
    B, R, S = src.shape
    if dst is None and dst_hi is None:
        dst = torch.empty(B, S, R, device=src.device, dtype=torch.float32)
    ld = R if dst_ld is None else dst_ld
    bs = S * ld if dst_batch_stride is None else dst_batch_stride
    _lib.call("pg_transpose", _ptr(src), B, R, S, R * S, _ptr(dst), _ptr(dst_hi), _ptr(dst_lo), bs, ld, _fmt(dst_hi), _ptr(range_flag), _stream())
    return dst


def conv_desc(kind, B, C_in, C_out, L_in, k, stride, pad, in_rows, in_ld, precision, L_out=None,
              out_rows=None, out_ld=None, taps_per_group=0, base_offset_mode=0, max_ctas=0, max_clips_per_tile=0, weights_mn_major=0, cta_pair=0,
              whole_clip=0):
    if L_out is None:
        L_out = (L_in - 1) * stride - 2 * pad + k if kind == PG_CONV_TRANSPOSE else (L_in + 2 * pad - k) // stride + 1
    return ConvDesc(kind, B, C_in, C_out, L_in, L_out, k, stride, pad, in_rows, in_ld,
                    L_out if out_rows is None else out_rows, C_out if out_ld is None else out_ld,
                    precision, taps_per_group, base_offset_mode, max_ctas, max_clips_per_tile, weights_mn_major, cta_pair, whole_clip)


def pack_weight(w, kind, want_tc=True, want_simt=False, plane_dtype=torch.bfloat16, want_lo=True):
    """torch Conv1d [C_out,C_in,k] / ConvTranspose1d [C_in,C_out,k] weight -> kernel layouts."""
    w = _need_cuda(w.detach(), "weight")
    if kind == PG_CONV_TRANSPOSE:
        C_in, C_out, k = w.shape
    else:
        C_out, C_in, k = w.shape
    hi = lo = simt = None
    if want_tc:
        hi = torch.empty(k, C_out, C_in, device=w.device, dtype=plane_dtype)
        lo = torch.empty_like(hi) if want_lo else None
    if want_simt:
        simt = torch.empty(k, C_in, C_out, device=w.device, dtype=torch.float32)
    _lib.call("pg_pack_weight", _ptr(w), kind, C_in, C_out, k, _ptr(hi), _ptr(lo), _ptr(simt), _fmt(hi), _stream())
    return hi, lo, simt


def conv_tc(desc, x_hi, x_lo, w_hi, w_lo, y, stats, epilogue=None, out_rows=None):
    """epilogue: a ConvEpilogue (conv_epilogue()) to fuse activation / per-clip norm + activation and the operand-plane
    writes into the kernel; None = raw fp32 output + statistics records.
    out_rows (ragged batch): int32 CUDA [B], the valid output rows of each clip (pg_conv_tc_ragged)."""
    if out_rows is not None:
        _lib.call("pg_conv_tc_ragged", C.byref(desc), _ptr(x_hi), _ptr(x_lo), _ptr(w_hi), _ptr(w_lo), _ptr(y), _ptr(stats),
                  C.byref(epilogue) if epilogue is not None else None, _ptr(_lengths(out_rows, desc.B, "out_rows")), _stream())
        return
    _lib.call("pg_conv_tc", C.byref(desc), _ptr(x_hi), _ptr(x_lo), _ptr(w_hi), _ptr(w_lo), _ptr(y), _ptr(stats),
              C.byref(epilogue) if epilogue is not None else None, _stream())


_NO_DST = ActDst(None, None, 0, 0, 0, PG_DT_NONE, 1.0, None)


def conv_epilogue(mode, dst0, dst1=None, gamma=None, beta=None, eps=1e-5, scale_shift=None):
    return ConvEpilogue(mode, gamma.data_ptr() if gamma is not None else None, beta.data_ptr() if beta is not None else None,
                        float(eps), dst0, dst1 if dst1 is not None else _NO_DST,
                        scale_shift.data_ptr() if scale_shift is not None else None)


def conv_epilogue_supported(desc, mode):
    r = _lib.load().pg_conv_epilogue_supported(C.byref(desc), mode)
    if r < 0:
        raise RuntimeError(f"pg_conv_epilogue_supported failed ({r}): {_lib.last_error()}")
    return bool(r)


def conv_stat_parts(desc):
    p = _lib.load().pg_conv_stat_parts(C.byref(desc))
    if p <= 0:
        raise RuntimeError(f"pg_conv_stat_parts failed ({p}): {_lib.last_error()}")
    return p


_PLAN_KEYS = ("n_tile", "n_ntiles", "nb", "strip_rows", "pair", "merged", "mgroups", "acc_stages", "n_chunks", "n_cotiles",
              "OS", "IS", "taps0", "taps1", "groups0", "groups1", "whole_clip")


def conv_plan(desc, whole_clip=None):
    """Host-side tiling plan of pg_conv_tc for a layer (pg_conv_tc_plan) as a dict, plus `tiles` and `units` (persistent
    CTAs or CTA pairs).  whole_clip: plan the whole-clip tiles of the fused per-clip norm epilogue; None if they do not fit."""
    d = ConvDesc.from_buffer_copy(desc)
    if whole_clip is not None:
        d.tc_whole_clip = int(whole_clip)
    out = (C.c_int * 17)()
    if _lib.load().pg_conv_tc_plan(C.byref(d), out, 17) != 0:
        return None
    pl = dict(zip(_PLAN_KEYS, out))
    slabs = pl["n_cotiles"] // 2 if pl["pair"] else pl["n_cotiles"]
    parts = 1 if pl["whole_clip"] else pl["OS"] * pl["n_ntiles"]
    pl["tiles"] = slabs * parts * -(-d.B // pl["nb"])
    pl["units"] = 74 if pl["pair"] else 148
    return pl


def conv_simt(desc, x, w_simt, y):
    _lib.call("pg_conv_simt", C.byref(desc), _ptr(x), _ptr(w_simt), _ptr(y), _stream())


def channel_stats(y, B, L, Cn, rows, ld, stats):
    _lib.call("pg_channel_stats", _ptr(y), B, L, Cn, rows, ld, _ptr(stats), _stream())


def bn_finalize(stats, B, P, Cn, per_clip, gamma, beta, eps, scale_shift, mean_var=None):
    _lib.call("pg_bn_finalize", _ptr(stats), B, P, Cn, int(per_clip), _ptr(gamma), _ptr(beta), eps,
              _ptr(scale_shift), _ptr(mean_var), _stream())


def act_dst(hi, lo, batch_stride, ld, ch_off, dtype, slope, range_flag=None):
    return ActDst(hi.data_ptr() if hi is not None else None, lo.data_ptr() if lo is not None else None,
                  batch_stride, ld, ch_off, dtype, slope, range_flag.data_ptr() if range_flag is not None else None)


def bn_running_update(mean_var, running_mean, running_var, momentum, unbias):
    """running = (1 - momentum) * running + momentum * batch statistic (variance times `unbias`), in place, one launch.
    mean_var: float32 [.., C, 2] as written by bn_finalize (its first group is used)."""
    Cn = running_mean.numel()
    for t, name in ((mean_var, "mean_var"), (running_mean, "running_mean"), (running_var, "running_var")):
        _need_cuda(t, name)
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise RuntimeError(f"phasegen.bn_running_update: {name} must be a contiguous float32 CUDA tensor")
    if mean_var.numel() < 2 * Cn or running_var.numel() != Cn:
        raise RuntimeError("phasegen.bn_running_update: shapes do not match")
    _lib.call("pg_bn_running_update", _ptr(mean_var), _ptr(running_mean), _ptr(running_var), Cn, float(momentum), float(unbias), _stream())


def bn_from_running(running_mean, running_var, gamma, beta, eps, scale_shift, mean_var=None):
    """eval-mode norm: (scale, shift) from the running statistics, replicated over the G rows of scale_shift [G, C, 2]."""
    G, Cn = scale_shift.shape[0], scale_shift.shape[1]
    _lib.call("pg_bn_from_running", _ptr(running_mean), _ptr(running_var), _ptr(gamma), _ptr(beta), float(eps), Cn, G,
              _ptr(scale_shift), _ptr(mean_var), _stream())


def bn_act(y, B, L, Cn, rows, ld, scale_shift, per_clip, dst0, dst1=None, clip_rows=None):
    """clip_rows (ragged batch): int32 CUDA [B], the valid rows of each clip; rows beyond them are written as 0."""
    if clip_rows is not None:
        _lib.call("pg_bn_act_ragged", _ptr(y), B, L, Cn, rows, ld, _ptr(scale_shift), int(per_clip),
                  C.byref(dst0), C.byref(dst1) if dst1 is not None else None, _ptr(_lengths(clip_rows, B, "clip_rows")), _stream())
        return
    _lib.call("pg_bn_act", _ptr(y), B, L, Cn, rows, ld, _ptr(scale_shift), int(per_clip),
              C.byref(dst0), C.byref(dst1) if dst1 is not None else None, _stream())


# ------------------------------------------------------------------------- training step
def grad_src(g, ld, ch_off, slope):
    return _lib.GradSrc(g.data_ptr(), ld, ch_off, slope)


def phase_loss(out_cl, logmag_cl, phase_cl, d_out, partial, loss3, mag_weight=0.2):
    """out [B,T,2C], targets [B,T,C] channels-last -> loss3 = (total, cos, sin, mag) and d_out."""
    B, T, C2 = out_cl.shape
    _lib.call("pg_phase_loss", _ptr(out_cl), _ptr(logmag_cl), _ptr(phase_cl), B * T, C2 // 2, mag_weight,
              _ptr(d_out), _ptr(partial), partial.shape[0], _ptr(loss3), _stream(), n_kernels=2)


def bn_bwd(z, B, L, Cn, scale_shift, mean_var, eps, g0, g1, partial, coef, dgamma, dbeta, dz_hi, dz_lo, dz_rows, dz_dtype):
    n_chunks = partial.shape[0] if partial is not None else 0
    _lib.call("pg_bn_bwd", _ptr(z), B, L, Cn, _ptr(scale_shift), _ptr(mean_var), eps, C.byref(g0),
              C.byref(g1) if g1 is not None else None, _ptr(partial), n_chunks, _ptr(coef), _ptr(dgamma), _ptr(dbeta),
              _ptr(dz_hi), _ptr(dz_lo), dz_rows, dz_dtype, _stream(), n_kernels=3 if scale_shift is not None else 1)


def wgrad_tc(desc, x_hi, x_lo, g_hi, g_lo, g_rows, dw_packed):
    dt = PG_DT_BF16 if dw_packed.dtype == torch.bfloat16 else PG_DT_F32
    _lib.call("pg_wgrad_tc", C.byref(desc), _ptr(x_hi), _ptr(x_lo), _ptr(g_hi), _ptr(g_lo), g_rows, _ptr(dw_packed), dt, _stream())


def wgrad_simt(desc, x, g, g_rows, dw_packed):
    _lib.call("pg_wgrad_simt", C.byref(desc), _ptr(x), _ptr(g), g_rows, _ptr(dw_packed), _stream())


def unpack_grad(packed, kind, out):
    k, C_out, C_in = packed.shape
    _lib.call("pg_unpack_grad", _ptr(packed), kind, C_in, C_out, k, _ptr(out), _stream())


def adam_step(p, g, m, v, lr, beta1, beta2, eps, step, grad_scale=1.0, w_hi=None, w_lo=None):
    gdt = PG_DT_BF16 if g.dtype == torch.bfloat16 else PG_DT_F32
    _lib.call("pg_adam_step", _ptr(p), _ptr(g), gdt, _ptr(m), _ptr(v), p.numel(), lr, beta1, beta2, eps, step, grad_scale,
              _ptr(w_hi), _ptr(w_lo), _stream())


def cast_split(src, hi, lo=None, range_flag=None):
    """fp32 (contiguous) -> bf16 or fp16 hi(/lo) planes of the same element order."""
    _lib.call("pg_cast_split", _ptr(src), src.numel(), _ptr(hi), _ptr(lo), _fmt(hi), _ptr(range_flag), _stream())


def packed_view(weight, kind):
    """The [k][C_out][C_in] view of a Conv1d / ConvTranspose1d weight if its memory already has that
    layout (the drop-in model stores its weights that way), else None."""
    w = weight.detach()
    v = w.permute(2, 1, 0) if kind == PG_CONV_TRANSPOSE else w.permute(2, 0, 1)
    return v if v.is_contiguous() else None


def to_packed_storage(weight, kind):
    """Re-lay a weight tensor so that its memory is [k][C_out][C_in] while its logical shape (and
    therefore state_dict / checkpoint format) stays the torch one."""
    w = weight.detach()
    packed = (w.permute(2, 1, 0) if kind == PG_CONV_TRANSPOSE else w.permute(2, 0, 1)).contiguous()
    return packed.permute(2, 1, 0) if kind == PG_CONV_TRANSPOSE else packed.permute(1, 2, 0)
