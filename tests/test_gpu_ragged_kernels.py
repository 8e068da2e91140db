"""The four ragged-batch entry points (pg_stft_ragged, pg_istft_ragged, pg_conv_tc_ragged, pg_bn_act_ragged) one by one,
clip by clip, against float64 references of the same operation, with per-clip tables built from adversarial lengths:
the full length, a length of 1 (or 0), lengths that end on a position-tile or CTA-run seam and one row either side of
it, odd lengths on stride-2 layers, and clips of very different lengths next to each other.  Everything a kernel must
not read holds NaN.  Tolerances are those of the fixed-shape tests (test_gpu_stft.py, test_gpu_conv.py)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import stft_np, unet_torch  # noqa: E402
from test_gpu_conv import GEOM, _case  # noqa: E402

CONV_TOL = {"bf16x3": 3e-5, "f16x3": 3e-5, "f16x2": 5e-4, "f16": 8e-4}
# the shape lists of test_tc_conv_cta_pairs and test_tc_conv_fused_epilogues
PAIR_SHAPES = [("d1", 128, 136, 3, 16), ("d2", 128, 69, 3, 16), ("d3", 128, 66, 5, 16), ("d4", 64, 31, 9, 16),
               ("u4", 128, 15, 9, 16), ("u3", 128, 31, 5, 16), ("u2", 128, 66, 3, 1), ("u1", 128, 69, 3, 16),
               ("u1", 128, 349, 40, 16), ("d1", 128, 696, 21, 16), ("d2", 128, 349, 24, 16), ("u4", 128, 85, 7, 16)]
FUSED_SHAPES = [("d1", 128, 696, 5, 0), ("d4", 128, 171, 7, 0), ("d1", 64, 136, 3, 1), ("d2", 128, 349, 5, 0),
                ("d3", 128, 346, 5, 0), ("u4", 128, 171, 5, 0), ("u3", 128, 171, 5, 0), ("u2", 128, 346, 5, 0),
                ("u2", 64, 346, 3, 1), ("u3", 64, 171, 6, 1), ("d3", 128, 66, 9, 0), ("u4", 128, 135, 9, 0),
                ("d2", 128, 69, 7, 0), ("u3", 128, 121, 5, 0)]


def rel_l2(a, b):
    dt = np.complex128 if (np.iscomplexobj(a) or np.iscomplexobj(b)) else np.float64
    a = np.asarray(a, dt); b = np.asarray(b, dt)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _i32(v):
    return torch.tensor([int(x) for x in v], dtype=torch.int32, device="cuda")


def _bits(t):
    return t.view(torch.int16)


# ------------------------------------------------------------------------------------------------------------ STFT
def _stft_call(wave, n_fft, n_b, T_b, fmt):
    """pg_stft_ragged -> (a, second, hi, lo): fmt None = general variant with the phase plane, else the inference
    variant writing 16-bit operand planes of that dtype."""
    from phasegen import ops
    B, N = wave.shape
    T, C = 1 + N // (n_fft // 4), n_fft // 2
    if fmt is None:
        a, ph = ops.stft(wave, n_fft, n_fft // 4, clip_samples=_i32(n_b), clip_frames=_i32(T_b))
        return a, ph, None, None
    hi = torch.full((B, T, C), 7.0, device="cuda", dtype=fmt); lo = torch.full_like(hi, 7.0)
    a, _ = ops.stft(wave, n_fft, n_fft // 4, want_second=False, operand=(hi, lo, T * C),
                    clip_samples=_i32(n_b), clip_frames=_i32(T_b))
    return a, None, hi, lo


def _check_stft(n_fft, T, clips, seed):
    """clips: (n_b, T_b).  Clip b is its first min(n_b, (T_b - 1)*hop) samples zero-padded to (T_b - 1)*hop; samples
    up to n_b are real, later ones NaN.  The call on a buffer whose base is 4 bytes past an 8-byte boundary (no float2
    loads) must give the same bits as on an aligned one."""
    hop = n_fft // 4
    N, B = (T - 1) * hop, len(clips)
    n_b, T_b = [c[0] for c in clips], [c[1] for c in clips]
    rng = np.random.default_rng(seed)
    w = (0.3 * rng.standard_normal((B, N)) + np.sin(0.05 * np.arange(N))).astype(np.float32)
    for b, n in enumerate(n_b):
        w[b, max(n, 0):] = np.nan
    aligned = torch.from_numpy(w).cuda()
    buf = torch.empty(B * N + 1, device="cuda")
    buf[1:] = aligned.reshape(-1)
    shifted = buf[1:].view(B, N)
    assert aligned.data_ptr() % 8 == 0 and shifted.data_ptr() % 8 == 4
    refs = []
    for b in range(B):
        x = np.zeros((T_b[b] - 1) * hop)
        m = min(n_b[b], x.size)
        x[:m] = w[b, :m]
        refs.append(stft_np.stft(x, n_fft, hop)[1:].T)       # [T_b, C], DC row dropped
    for fmt in (None, torch.bfloat16, torch.float16):
        outs = [_stft_call(wv, n_fft, n_b, T_b, fmt) for wv in (aligned, shifted)]
        for u, v in zip(*outs):
            if u is not None:
                assert torch.equal(u.view(torch.int32) if u.dtype == torch.float32 else _bits(u),
                                   v.view(torch.int32) if v.dtype == torch.float32 else _bits(v)), ("alignment", fmt)
        a, ph, hi, lo = outs[0]
        for b in range(B):
            S = refs[b]
            assert rel_l2(a[b, :T_b[b]].cpu().numpy(), np.log1p(np.abs(S))) < 1e-4, (fmt, b, n_b[b], T_b[b])
            assert not bool(a[b, T_b[b]:].view(torch.int32).any()), (fmt, b, "frames >= T_b")
            if ph is not None:
                z = np.abs(S) * np.exp(1j * ph[b, :T_b[b]].cpu().numpy().astype(np.float64))
                assert rel_l2(z, S) < 1e-4, (b, "phase")         # |S|-weighted, as in test_stft_matches_oracle
                assert not bool(ph[b, T_b[b]:].any()), (b, "phase frames >= T_b")     # atan2 of zeros: +0 or -0
        if hi is not None:
            want_hi = a.to(fmt)
            want_lo = (a - want_hi.float()).to(fmt)
            assert torch.equal(_bits(hi), _bits(want_hi)) and torch.equal(_bits(lo), _bits(want_lo)), fmt


@pytest.mark.parametrize("n_fft", [256, 512, 1024, 2048])
def test_stft_ragged_matches_the_oracle_per_clip(n_fft):
    hop = n_fft // 4
    fpc = 4 * 256 // (n_fft // 32)                              # frames per CTA
    T = fpc + 8
    clips = [((T - 1) * hop, T),                                # the full buffer
             (fpc * hop, fpc + 1),                              # n_b == (T_b - 1)*hop, one frame past a CTA's run
             ((fpc - 1) * hop - 1, fpc),                        # one sample short, T_b on the CTA seam
             ((fpc - 2) * hop - (hop - 1), fpc - 1),            # hop - 1 samples short, one frame before the seam
             (9 * hop + hop // 3, 12),                          # not a multiple of hop
             (n_fft // 2 + 1, 4),                               # the shortest clip: every frame reflects
             (hop + 5, 4)]
    _check_stft(n_fft, T, clips, seed=n_fft)


@pytest.mark.parametrize("n_fft", [256, 512, 1024, 2048])
def test_stft_ragged_reads_a_clip_only_up_to_its_padded_end(n_fft):
    """A table with n_b > (T_b - 1)*hop + 3*hop: clip b is still its first (T_b - 1)*hop samples, frames >= T_b stay 0,
    and the result does not depend on the buffer's alignment."""
    hop = n_fft // 4
    T = 4 * 256 // (n_fft // 32) + 8
    N = (T - 1) * hop
    clips = [((T - 6) * hop + 5, T - 8), (N, 4), (N - 3, T // 2), (N, T)]
    assert all(n > (t - 1) * hop + 3 * hop for n, t in clips[:3])
    _check_stft(n_fft, T, clips, seed=n_fft + 1)


# ----------------------------------------------------------------------------------------------------------- ISTFT
@pytest.mark.parametrize("mode", ["polar_log", "cartesian"])
@pytest.mark.parametrize("n_fft,T", [(1024, 87), (1024, 171), (512, 171)])
def test_istft_ragged_matches_the_oracle_per_clip(n_fft, T, mode):
    """T_b of 2, 3, 86 and 87 around the 85-hop-block CTA run, per-clip (scale, shift) of the second plane, NaN in every
    frame >= T_b; then NaN inside two clips' frames sets those clips' flags only."""
    from phasegen import ops
    hop, C = n_fft // 4, n_fft // 2
    clips = [(T, (T - 1) * hop), (2, hop - 3), (3, 2 * hop), (86, 85 * hop - 1), (87, 86 * hop - hop // 2 - 1), (86, 2 * hop + 1)]
    B = len(clips)
    rng = np.random.default_rng(T + n_fft)
    if mode == "polar_log":
        a = np.abs(rng.standard_normal((B, T, C))); b = 3.0 * rng.standard_normal((B, T, C))
    else:
        a = rng.standard_normal((B, T, C)); b = rng.standard_normal((B, T, C))
    a, b = a.astype(np.float32), b.astype(np.float32)
    ss = np.stack([1.0 + 0.2 * rng.standard_normal((B, C)), 0.3 * rng.standard_normal((B, C))], -1).astype(np.float32)
    for i, (T_b, _) in enumerate(clips):
        a[i, T_b:] = np.nan; b[i, T_b:] = np.nan
    spec = ops.PG_SPEC_POLAR_LOG if mode == "polar_log" else ops.PG_SPEC_CARTESIAN
    ta, tb, tss = (torch.from_numpy(v).cuda() for v in (a, b, ss))
    frames, samples = _i32([c[0] for c in clips]), _i32([c[1] for c in clips])
    bad = torch.full((B,), 5, device="cuda", dtype=torch.int32)
    wv, peak = ops.istft(ta, tb, spec, n_fft, hop, normalize=False, check_finite=False, b_scale_shift=tss, bad_out=bad,
                         clip_frames=frames, clip_samples=samples)
    assert bad.tolist() == [0] * B
    for i, (T_b, n) in enumerate(clips):
        bb = b[i, :T_b].astype(np.float64) * ss[i, :, 0] + ss[i, :, 1]
        z = stft_np.polar_to_complex(a[i, :T_b], bb) if mode == "polar_log" else a[i, :T_b].astype(np.float64) + 1j * bb
        ref = stft_np.istft(np.concatenate([np.zeros((1, T_b)), z.T]), hop)
        got = wv[i].cpu().numpy()
        assert rel_l2(got[:n], ref[:n]) < 2e-5, (i, T_b, n)
        assert not got[n:].any(), (i, "samples >= n_b")
        assert abs(float(peak[i]) - np.abs(ref).max()) < 1e-4 * np.abs(ref).max(), (i, "peak")
    ta[2, 1, 5] = float("nan")                                  # inside clip 2 (T_b = 3)
    tb[3, 85, 7] = float("nan")                                 # clip 3's last frame (T_b = 86)
    ops.istft(ta, tb, spec, n_fft, hop, normalize=False, check_finite=False, b_scale_shift=tss, bad_out=bad,
              clip_frames=frames, clip_samples=samples)
    assert bad.tolist() == [0, 0, 1, 1, 0, 0]


# ----------------------------------------------------------------------------------------------------- convolution
def _out_len(kind, k, s, p, L):
    return (L - 1) * s - 2 * p + k if kind else (L + 2 * p - k) // s + 1


def _conv_clips(layer, L_in, L_out, seam, B):
    """(L_in_b, L_b) per clip: L_b from the layer's length rule for a shortened input, or an arbitrary L_b <= L_out on a
    full input (position-tile seam and one row either side, one row), cycled over the batch so that neighbours in a
    merged tile get very different lengths."""
    kind, k, s, p = GEOM[layer][:4]
    rule = lambda L: (L, min(L_out, max(0, _out_len(kind, k, s, p, L))))
    cands = [(L_in, L_out), (L_in, seam), rule(1), (L_in, seam - 1), rule(max(1, L_in // 3) | 1),
             (L_in, min(seam + 1, L_out)), rule(L_in - 1), (L_in, 1), rule(2), (L_in, L_out - 1)]
    return [cands[i % len(cands)] for i in range(B)]


def _conv_setup(layer, C, L_in, B, seed):
    """Input with rows >= L_in_b zero (the executor's invariant), the per-clip table and the float64 reference."""
    from phasegen import ops
    kind, k, s, p, C_in, C_out, rows, x, w = _case(layer, C, L_in, B, seed=seed)
    L_out = _out_len(kind, k, s, p, L_in)
    d = ops.conv_desc(kind, B, C_in, C_out, L_in, k, s, p, rows, C_in, ops.PG_PREC_BF16X3, taps_per_group=16)
    pl = ops.conv_plan(d)
    seam = pl["OS"] * pl["n_tile"]                              # first output row of the second position tile
    if seam >= L_out:
        seam = L_out // 2 | 1
    clips = _conv_clips(layer, L_in, L_out, seam, B)
    for b, (L_in_b, _) in enumerate(clips):
        x[b, L_in_b:] = 0
    xd = x[:, :L_in].double().permute(0, 2, 1).cpu()
    ref = (F.conv_transpose1d if kind else F.conv1d)(xd, w.double().cpu(), None, s, p).permute(0, 2, 1)
    return kind, k, s, p, C_in, C_out, rows, x, w, L_out, [c[1] for c in clips], ref


def _planes(x, pdt):
    xh = x.to(pdt)
    return xh, (x - xh.float()).to(pdt)


@pytest.mark.parametrize("layer,C,L_in,B,tpg", PAIR_SHAPES)
def test_conv_tc_ragged_raw_output_and_statistics(layer, C, L_in, B, tpg):
    """PG_EPI_RAW on single CTAs and CTA pairs (cta_pair 0, 1, 2), four precisions: rows < L_b match float64, the
    statistics records count exactly L_b rows per (clip, channel) and their combined moments are those of rows < L_b."""
    from phasegen import ops
    from phasegen._lib import PRECISIONS
    kind, k, s, p, C_in, C_out, rows, x, w, L_out, L_b, ref = _conv_setup(layer, C, L_in, B, seed=21)
    for prec in ("bf16x3", "f16x3", "f16x2", "f16"):
        pdt = torch.float16 if prec.startswith("f16") else torch.bfloat16
        whi, wlo, _ = ops.pack_weight(w, kind, plane_dtype=pdt)
        xh, xl = _planes(x, pdt)
        for pair in (0, 1, 2):
            d = ops.conv_desc(kind, B, C_in, C_out, L_in, k, s, p, rows, C_in, PRECISIONS[prec], taps_per_group=tpg,
                              cta_pair=pair)
            y = torch.full((B, L_out, C_out), float("nan"), device="cuda")
            st = torch.zeros(B, ops.conv_stat_parts(d), C_out, 4, device="cuda")
            ops.conv_tc(d, xh, xl if prec != "f16" else None, whi, wlo if prec.endswith("x3") else None, y, st,
                        out_rows=_i32(L_b))
            yc, stc = y.double().cpu(), st.double().cpu()
            n = stc[..., 0].sum(1)
            for b in range(B):
                tag = (layer, prec, pair, b, L_b[b])
                assert bool((n[b] == L_b[b]).all()), tag
                if L_b[b] == 0:
                    continue
                yb = yc[b, :L_b[b]]
                assert rel_l2(yb, ref[b, :L_b[b]]) < CONV_TOL[prec], tag
                mean = (stc[b, :, :, 0] * stc[b, :, :, 1]).sum(0) / n[b]
                m2 = (stc[b, :, :, 2] + stc[b, :, :, 0] * (stc[b, :, :, 1] - mean) ** 2).sum(0)
                assert float((mean - yb.mean(0)).abs().max()) < 1e-4, tag
                var = yb.var(0, unbiased=False)
                assert float((m2 / n[b] - var).abs().max()) < 1e-4 * max(float(var.max()), 1e-6), tag


@pytest.mark.parametrize("layer,C,L_in,B,pair", FUSED_SHAPES)
def test_conv_tc_ragged_fused_epilogues(layer, C, L_in, B, pair):
    """PG_EPI_ACT (d1, d4) and PG_EPI_NORM_ACT (whole-clip tiles): the per-clip norm over rows < L_b, the affine and
    LeakyReLU(0.2) / ReLU into two destinations, the second at a channel offset of a wider buffer; exact zeros in rows
    [L_b, L_out); nothing written outside rows < L_out and the destination's channels; no range flag."""
    from phasegen import ops
    from phasegen._lib import PG_DT_BF16_SPLIT, PG_DT_F16_SPLIT, PG_EPI_ACT, PG_EPI_NORM_ACT, PRECISIONS
    kind, k, s, p, C_in, C_out, rows, x, w, L_out, L_b, ref = _conv_setup(layer, C, L_in, B, seed=22)
    has_norm = layer not in ("d1", "d4")
    mode = PG_EPI_NORM_ACT if has_norm else PG_EPI_ACT
    g = torch.Generator().manual_seed(23)
    gamma = (1.0 + 0.2 * torch.randn(C_out, generator=g)).cuda()
    beta = (0.3 * torch.randn(C_out, generator=g)).cuda()
    rows_o, wide, off, SENT = (L_out + 7) // 8 * 8, 2 * C_out, C_out, 7.0
    for prec in ("bf16x3", "f16x3", "f16x2"):
        f16 = prec.startswith("f16")
        pdt = torch.float16 if f16 else torch.bfloat16
        d = ops.conv_desc(kind, B, C_in, C_out, L_in, k, s, p, rows, C_in, PRECISIONS[prec], taps_per_group=16, cta_pair=pair)
        if not ops.conv_epilogue_supported(d, mode):
            assert (layer, pair, L_in) == ("u2", 1, 346)        # as in test_tc_conv_fused_epilogues
            continue
        whi, wlo, _ = ops.pack_weight(w, kind, plane_dtype=pdt)
        xh, xl = _planes(x, pdt)
        dt = PG_DT_F16_SPLIT if f16 else PG_DT_BF16_SPLIT
        flag = torch.zeros(1, device="cuda", dtype=torch.int32)
        a_hi = torch.full((B, rows_o, C_out), SENT, device="cuda", dtype=pdt); a_lo = torch.full_like(a_hi, SENT)
        c_hi = torch.full((B, rows_o, wide), SENT, device="cuda", dtype=pdt); c_lo = torch.full_like(c_hi, SENT)
        epi = ops.conv_epilogue(mode, ops.act_dst(a_hi, a_lo, rows_o * C_out, C_out, 0, dt, 0.2, flag),
                                ops.act_dst(c_hi, c_lo, rows_o * wide, wide, off, dt, 0.0, flag),
                                gamma if has_norm else None, beta if has_norm else None, 1e-5)
        ops.conv_tc(d, xh, xl, whi, wlo if prec.endswith("x3") else None, None, None, epi, out_rows=_i32(L_b))
        tol = 2e-3 if prec == "f16x2" else 2e-4
        got_a = (a_hi.double() + a_lo.double()).cpu()
        got_c = (c_hi.double() + c_lo.double()).cpu()
        for b in range(B):
            tag = (layer, prec, pair, b, L_b[b])
            if L_b[b]:
                h = ref[b, :L_b[b]]
                if has_norm:
                    mean, var = h.mean(0), h.var(0, unbiased=False)
                    h = (h - mean) / torch.sqrt(var + 1e-5) * gamma.double().cpu() + beta.double().cpu()
                assert rel_l2(got_a[b, :L_b[b]], torch.where(h > 0, h, 0.2 * h)) < tol, tag + ("leaky",)
                assert rel_l2(got_c[b, :L_b[b], off:], h.clamp(min=0)) < tol, tag + ("relu at a channel offset",)
            for t in (a_hi, a_lo):
                assert not bool(t[b, L_b[b]:L_out].float().any()), tag + ("rows >= L_b",)
            for t in (c_hi, c_lo):
                assert not bool(t[b, L_b[b]:L_out, off:].float().any()), tag + ("rows >= L_b",)
        for t in (a_hi, a_lo, c_hi, c_lo):
            assert bool((t[:, L_out:] == SENT).all()), (layer, prec, "rows >= L_out")
        assert bool((c_hi[:, :, :off] == SENT).all() and (c_lo[:, :, :off] == SENT).all()), (layer, prec, "channels")
        assert int(flag.item()) == 0, (layer, prec)


# ---------------------------------------------------------------------------------------------------------- bn_act
def test_bn_act_ragged_zeroes_rows_past_each_clip():
    """Per-clip (scale, shift), an fp16-split destination and a bf16-split one at a channel offset; y holds 1e6 and NaN
    past every L_b: those rows must come out as exact zeros and the fp16 range flag must stay 0."""
    from phasegen import ops
    from phasegen._lib import PG_DT_BF16_SPLIT, PG_DT_F16_SPLIT
    B, L, rows, Cn = 6, 45, 48, 128
    L_b = [L, 0, 1, 17, L - 1, 30]
    g = torch.Generator().manual_seed(31)
    y = torch.randn(B, rows, Cn, generator=g)
    for b, n in enumerate(L_b):
        y[b, n:, 0::2] = 1.0e6
        y[b, n:, 1::2] = float("nan")
    ss = torch.stack([1.0 + 0.2 * torch.randn(B, Cn, generator=g), 0.3 * torch.randn(B, Cn, generator=g)], -1)
    flag = torch.zeros(1, device="cuda", dtype=torch.int32)
    SENT = 7.0
    h0 = torch.full((B, rows, Cn), SENT, device="cuda", dtype=torch.float16); l0 = torch.full_like(h0, SENT)
    h1 = torch.full((B, rows, 2 * Cn), SENT, device="cuda", dtype=torch.bfloat16); l1 = torch.full_like(h1, SENT)
    ops.bn_act(y.cuda(), B, L, Cn, rows, Cn, ss.cuda(), True, ops.act_dst(h0, l0, rows * Cn, Cn, 0, PG_DT_F16_SPLIT, 0.2, flag),
               ops.act_dst(h1, l1, rows * 2 * Cn, 2 * Cn, Cn, PG_DT_BF16_SPLIT, 0.0, flag), clip_rows=_i32(L_b))
    assert int(flag.item()) == 0
    got0 = (h0.double() + l0.double()).cpu(); got1 = (h1.double() + l1.double()).cpu()
    for b, n in enumerate(L_b):
        z = y[b, :n].double() * ss[b, :, 0].double() + ss[b, :, 1].double()
        if n:
            assert rel_l2(got0[b, :n], torch.where(z > 0, z, 0.2 * z)) < 2e-4, b
            assert rel_l2(got1[b, :n, Cn:], z.clamp(min=0)) < 2e-4, b
        assert not bool(got0[b, n:L].any()) and not bool(got1[b, n:L, Cn:].any()), (b, "rows >= L_b")
    for t in (h0, l0, h1, l1):
        assert bool((t[:, L:] == SENT).all())
    assert bool((h1[:, :, :Cn] == SENT).all() and (l1[:, :, :Cn] == SENT).all())


# -------------------------------------------------------------------------------------------------------- bad tables
def test_bad_tables_stay_inside_their_buffers():
    """Table entries a little out of range (past the extent, 0, -1).  Every buffer a kernel reads or writes sits inside a
    sentinel guard wide enough that an unclamped kernel would still touch only the guard; the guards must be intact
    and each result must equal the call with the table clamped to [0, extent]."""
    from phasegen import ops
    from phasegen._lib import PG_DT_BF16_SPLIT, PG_EPI_NORM_ACT, PG_SPEC_CARTESIAN, PRECISIONS
    G, SENT, SENT16 = 8192, 12345.0, 7.0                       # 7 is exact in bf16 and fp16

    def guarded(shape, fill=SENT, dtype=torch.float32):
        n = int(np.prod(shape))
        buf = torch.full((n + 2 * G,), fill, device="cuda", dtype=dtype)
        return buf, buf[G:G + n].view(*shape)

    def intact(buf, view, fill=SENT):
        n = view.numel()
        edge = torch.cat([buf[:G], buf[G + n:]])
        return bool(torch.isnan(edge).all()) if fill != fill else bool((edge == fill).all())

    clamp = lambda v, hi: [min(max(int(x), 0), hi) for x in v]
    # STFT: the last clip's n_b runs past the buffer, the first clip's T_b past the frame count
    n_fft, T, B = 256, 40, 5
    hop, C = n_fft // 4, n_fft // 2
    N = (T - 1) * hop
    wbuf, wave = guarded((B, N), float("nan"))
    wave.copy_(torch.randn(B, N, device="cuda"))
    n_b, T_b = [N, 0, -1, 300, N + hop], [T + 3, T, 10, 0, -1]
    outs = []
    for ns, ts in ((n_b, T_b), (clamp(n_b, N), clamp(T_b, T))):
        abuf, a = guarded((B, T, C))
        hbuf, hi = guarded((B, T, C), SENT16, torch.bfloat16); lbuf, lo = guarded((B, T, C), SENT16, torch.bfloat16)
        cs, cf = _i32(ns), _i32(ts)                             # held: a dropped table's memory would be reused by the next
        ops._lib.call("pg_stft_ragged", ops._ptr(wave), B, N, n_fft, hop, ops._ptr(ops.twiddle(n_fft, wave.device)),
                      ops.PG_STFT_LOGMAG, ops._ptr(a), None, ops._ptr(hi), ops._ptr(lo), T * C, ops.PG_FMT_BF16,
                      ops._ptr(cs), ops._ptr(cf), ops._stream())
        assert intact(abuf, a) and intact(hbuf, hi, SENT16) and intact(lbuf, lo, SENT16)
        outs.append((a.clone(), hi.clone(), lo.clone()))
    assert intact(wbuf, wave, float("nan")) and bool(torch.isfinite(outs[0][0]).all())
    assert all(torch.equal(u.view(torch.int32) if u.dtype == torch.float32 else _bits(u),
                           v.view(torch.int32) if v.dtype == torch.float32 else _bits(v)) for u, v in zip(*outs))
    # ISTFT: the last clip's T_b runs past the input planes
    abuf, a = guarded((B, T, C), float("nan")); bbuf, bq = guarded((B, T, C), float("nan"))
    a.copy_(torch.randn(B, T, C, device="cuda")); bq.copy_(torch.randn(B, T, C, device="cuda"))
    T_b, n_b = [T, 0, -1, 10, T + 3], [N + hop, 0, 5 * hop, -1, N]
    outs = []
    for ts, ns in ((T_b, n_b), (clamp(T_b, T), clamp(n_b, N))):
        obuf, out = guarded((B, N))
        bad = torch.zeros(B, device="cuda", dtype=torch.int32)
        _, peak = ops.istft(a, bq, PG_SPEC_CARTESIAN, n_fft, hop, normalize=False, check_finite=False, out=out, bad_out=bad,
                            clip_frames=_i32(ts), clip_samples=_i32(ns))
        assert intact(obuf, out)
        outs.append((out.clone(), peak.clone(), bad.clone()))
    assert intact(abuf, a, float("nan")) and intact(bbuf, bq, float("nan"))
    assert outs[0][2].tolist() == [0] * B and all(torch.equal(u, v) for u, v in zip(*outs))
    # convolution, raw output + statistics and the fused per-clip norm: the last clip's L_b runs past L_out
    layer, Cc, L_in, Bc = "d3", 128, 66, 5
    kind, k, s, p, C_in, C_out, rows, x, w = _case(layer, Cc, L_in, Bc, seed=41)
    d = ops.conv_desc(kind, Bc, C_in, C_out, L_in, k, s, p, rows, C_in, PRECISIONS["bf16x3"], taps_per_group=16)
    L_out = d.L_out
    whi, wlo, _ = ops.pack_weight(w, kind)
    xh, xl = _planes(x, torch.bfloat16)
    L_b = [L_out, 0, -1, 7, L_out + 8]
    gamma = torch.ones(C_out, device="cuda"); beta = torch.zeros(C_out, device="cuda")
    outs = []
    for ls in (L_b, clamp(L_b, L_out)):
        ybuf, y = guarded((Bc, L_out, C_out))
        sbuf, st = guarded((Bc, ops.conv_stat_parts(d), C_out, 4))
        ops.conv_tc(d, xh, xl, whi, wlo, y, st, out_rows=_i32(ls))
        assert intact(ybuf, y) and intact(sbuf, st)
        rows_o = (L_out + 7) // 8 * 8
        hbuf, ah = guarded((Bc, rows_o, C_out), SENT16, torch.bfloat16)
        lbuf, al = guarded((Bc, rows_o, C_out), SENT16, torch.bfloat16)
        epi = ops.conv_epilogue(PG_EPI_NORM_ACT, ops.act_dst(ah, al, rows_o * C_out, C_out, 0, PG_DT_BF16_SPLIT, 0.2),
                                None, gamma, beta, 1e-5)
        ops.conv_tc(d, xh, xl, whi, wlo, None, None, epi, out_rows=_i32(ls))
        assert intact(hbuf, ah, SENT16) and intact(lbuf, al, SENT16)
        outs.append(([y[b, :n].clone() for b, n in enumerate(clamp(ls, L_out))], st.clone(), ah.clone(), al.clone()))
    assert all(torch.equal(u, v) for u, v in zip(outs[0][0], outs[1][0]))
    assert torch.equal(outs[0][1], outs[1][1]) and torch.equal(_bits(outs[0][2]), _bits(outs[1][2])) and \
        torch.equal(_bits(outs[0][3]), _bits(outs[1][3]))
    # bn_act
    Lr, Cn = 20, 64
    yv = torch.randn(Bc, Lr, Cn, device="cuda")
    L_b = [Lr + 8, 0, -1, 3, Lr]
    outs = []
    for ls in (L_b, clamp(L_b, Lr)):
        dbuf, dst = guarded((Bc, Lr, Cn))
        ops.bn_act(yv, Bc, Lr, Cn, Lr, Cn, None, False, ops.act_dst(dst, None, Lr * Cn, Cn, 0, ops.PG_DT_F32, 1.0),
                   clip_rows=_i32(ls))
        assert intact(dbuf, dst)
        outs.append(dst.clone())
    assert torch.equal(outs[0], outs[1])


# --------------------------------------------------------------------------------------------- executor, per layer
@pytest.mark.parametrize("prec", ["bf16x3", "f16mix1"])
def test_executor_layers_match_the_oracle_per_clip(prec):
    """UNetExecutor.run(clip_rows=...) at n_fft 512, B 6: every operand buffer (x0, a[i], cat[i], as hi + lo) and the
    final output, over rows < L_b of each clip, against the float64 oracle's per-layer taps of that clip alone, through
    the activation the buffer holds; rows [L_b, rows) are zero."""
    import model
    from phasegen import synth
    from phasegen.unet import clip_rows_table, layer_lengths
    n_fft, T = 512, 96
    C = n_fft // 2
    T_b = [T, 24, 88, 32, 48, 24]
    B = len(T_b)
    torch.manual_seed(51)
    net = model.UNetModel(C, 2 * C).cuda()
    synth.randomize_norm_affine(net, seed=52)
    sd = {k: v.detach().cpu() for k, v in net.model.state_dict().items()}
    g = torch.Generator().manual_seed(53)
    x = torch.log1p(torch.randn(B, T, C, generator=g).abs() * 2.0)
    for b, t in enumerate(T_b):
        x[b, t:] = 0
    levels = net._levels()
    ex = net.executor(B, T, "cuda", per_clip=True, phase_only=True, precision=prec)
    ex.load_input_cl(x.cuda())
    dn, up = net._norm_params(torch.device("cuda"))
    table = torch.tensor(clip_rows_table(levels, T_b), dtype=torch.int32, device="cuda")
    out = net._run(ex, dn, up, clip_rows=table).clone()
    lrelu, relu = (lambda t: F.leaky_relu(t, 0.2)), F.relu
    tol = 1e-3                                                  # the oracle bound on the predicted phase
    for b, t in enumerate(T_b):
        taps = {}
        unet_torch.unet_forward(sd, x[b:b + 1, :t].permute(0, 2, 1), torch.float64, per_clip_bn=True, taps=taps)
        cl = {k: v[0].T for k, v in taps.items()}               # [L, C] of this clip
        Ls = layer_lengths(levels, t)
        want = [("x0", ex.x0, Ls[0], x[b, :t].double()),
                ("a0", ex.a[0], Ls[1], lrelu(cl["y1"])), ("a1", ex.a[1], Ls[2], lrelu(cl["h2"])),
                ("a2", ex.a[2], Ls[3], lrelu(cl["h3"])), ("a3", ex.a[3], Ls[4], relu(cl["y4"])),
                ("cat0", ex.cat[0], Ls[1], relu(torch.cat([cl["y1"], cl["g2"]], 1))),
                ("cat1", ex.cat[1], Ls[2], relu(torch.cat([cl["h2"], cl["g3"]], 1))),
                ("cat2", ex.cat[2], Ls[3], relu(torch.cat([cl["h3"], cl["g4"]], 1)))]
        for name, op, L_b, ref in want:
            v = op.hi.double() + (op.lo.double() if op.lo is not None else 0)
            e =rel_l2(v[b, :L_b].cpu(), ref)
            assert e < tol, f"layer {name}, clip {b} (T_b {t}, L_b {L_b}): rel-L2 {e:.2e}"
            for plane in (op.hi, op.lo):
                if plane is not None:
                    assert not bool(plane[b, L_b:].float().any()), f"layer {name}, clip {b}: rows [{L_b}, {op.rows}) not zero"
        e = rel_l2(out[b, :Ls[-1]].cpu(), cl["out"][:, :C])
        assert e < tol, f"layer u1 (output), clip {b} (T_b {t}): rel-L2 {e:.2e}"
        assert not bool(out[b, Ls[-1]:].any()), f"layer u1 (output), clip {b}: rows past {Ls[-1]} not zero"
