"""Packed clips on the GPU: clips laid end to end in one flat buffer (PhaseGenPipeline.packed, run_host_packed), each clip
bit-identical to the ragged call on the padded [B, (T - 1)*hop] buffer that holds it in row b."""
import itertools

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import stft_np, unet_torch  # noqa: E402


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def snr_db(ref, est):
    ref = np.asarray(ref, np.float64); est = np.asarray(est, np.float64)
    g = np.dot(ref, est) / max(np.dot(est, est), 1e-300)
    return 10 * np.log10(np.sum(ref ** 2) / np.sum((ref - g * est) ** 2))


def _net(n_fft, seed):
    import model
    from phasegen import synth
    torch.manual_seed(seed)
    net = model.UNetModel(n_fft // 2, n_fft).cuda()
    synth.randomize_norm_affine(net, seed=seed + 1)
    return net


def _lengths(hop, N, seed):
    """The ragged suite's six lengths (full buffer, 24-frame minimum, a pair 8 frames apart), the one that is not a
    multiple of hop first and made odd, so the packed offsets include odd ones and ones that are 2 mod 4."""
    rng = np.random.default_rng(seed)
    n_min = 15 * hop + 1
    a = int(rng.integers(40 * hop, N - 16 * hop))
    n = [N, n_min, int(rng.integers(n_min, N)) // hop * hop + int(rng.integers(1, hop)), a, a - 8 * hop, int(rng.integers(n_min, N))]
    return [n[2] | 1] + n[:2] + n[3:]


def _full_lengths(B, sr, hop, seed):
    """B clips of 1 s to 4 s, the first not a multiple of hop and odd."""
    rng = np.random.default_rng(seed)
    n = [int(v) for v in rng.integers(sr, 4 * sr + 1, B)]
    n[0] = n[0] // hop * hop + 2 * int(rng.integers(0, hop // 2)) + 1
    return n


def _offsets(lengths):
    return list(itertools.accumulate([0] + list(lengths)))


def _padded_and_flat(B, N, lengths, sr, seed):
    """The ragged call's [B, N] buffer (NaN past every length: never read) and the same clips packed."""
    from phasegen import synth
    wave = synth.synthetic_waves(B, N, sr=sr, seed=seed, device="cuda")
    flat = torch.cat([wave[b, :n] for b, n in enumerate(lengths)]).contiguous()
    for b, n in enumerate(lengths):
        wave[b, n:] = float("nan")
    return wave, flat


def _assert_clips_equal(flat_out, padded_out, lengths):
    offs = _offsets(lengths)
    for b, n in enumerate(lengths):
        assert torch.equal(flat_out[offs[b]:offs[b + 1]], padded_out[b, :n]), b


@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("prec", ["bf16x3", "f16mix1"])
@pytest.mark.parametrize("n_fft,T,B", [(256, 64, 6), (1024, 696, 48)])
def test_packed_call_is_bit_identical_to_the_ragged_call(n_fft, T, B, prec, normalize):
    from phasegen.pipeline import PhaseGenPipeline, ragged_frames
    hop = n_fft // 4
    N = (T - 1) * hop
    sr = 16000 if n_fft == 256 else 44100
    lengths = _lengths(hop, N, seed=n_fft) if B == 6 else _full_lengths(B, sr, hop, seed=131)
    offs = _offsets(lengths)
    assert any(o % 2 for o in offs) and any(o % 4 == 2 for o in offs)
    pipe = PhaseGenPipeline(_net(n_fft, 141), n_fft, hop, precision=prec, per_clip=True, phase_only=True, normalize=normalize)
    wave, flat = _padded_and_flat(B, N, lengths, sr, seed=142)
    ragged = [t.clone() for t in pipe(wave, check_finite=True, return_intermediates=True, lengths=lengths)]
    audio, logmag, phase = pipe.packed(flat, lengths, frames=T, check_finite=True, return_intermediates=True)
    assert audio.shape == flat.shape and logmag.shape == ragged[1].shape
    _assert_clips_equal(audio, ragged[0], lengths)
    assert torch.equal(logmag, ragged[1]) and torch.equal(phase, ragged[2])
    assert pipe.nonfinite_clips(B) == []
    if ragged_frames(max(lengths), hop) == T:             # the default frame count is that of the longest clip
        assert torch.equal(pipe.packed(flat, lengths), audio)


def test_neighbours_do_not_reach_a_clip():
    from phasegen.pipeline import PhaseGenPipeline
    n_fft, T, B = 256, 64, 6
    hop = n_fft // 4
    lengths = _lengths(hop, (T - 1) * hop, seed=151)
    offs = _offsets(lengths)
    pipe = PhaseGenPipeline(_net(n_fft, 152), n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    _, flat = _padded_and_flat(B, (T - 1) * hop, lengths, 16000, seed=153)
    want = pipe.packed(flat, lengths).clone()
    for b in (1, 3):                                        # clip 2 (odd offset) and clip 4, each between NaN neighbours
        dirty = flat.clone()
        dirty[offs[b - 1]:offs[b]] = float("nan")
        dirty[offs[b + 1]:offs[b + 2]] = float("nan")
        got = pipe.packed(dirty, lengths)
        clip = got[offs[b]:offs[b + 1]]
        assert torch.equal(clip, want[offs[b]:offs[b + 1]]) and bool(torch.isfinite(clip).all()), b


def test_writes_stay_inside_the_output_view():
    from phasegen.pipeline import PhaseGenPipeline
    n_fft, T, B = 256, 64, 6
    hop = n_fft // 4
    lengths = _lengths(hop, (T - 1) * hop, seed=161)
    n = sum(lengths)
    pipe = PhaseGenPipeline(_net(n_fft, 162), n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    _, flat = _padded_and_flat(B, (T - 1) * hop, lengths, 16000, seed=163)
    want = pipe.packed(flat, lengths).clone()
    G = 1027                                                # the view starts 12 bytes past a 16-byte boundary
    big = torch.full((n + 2 * G,), -7.0, device="cuda")
    out = big[G:G + n]
    got = pipe.packed(flat, lengths, out=out)
    assert got.data_ptr() == out.data_ptr() and torch.equal(out, want)
    assert bool((big[:G] == -7.0).all()) and bool((big[G + n:] == -7.0).all())
    with pytest.raises(RuntimeError, match="out"):
        pipe.packed(flat, lengths, out=big[:n + 1])


def test_a_bad_offset_table_is_clamped_to_the_buffers():
    """Offsets beyond n_dst / n_wave: the kernels clamp them, so the guard around the views keeps its sentinel (an
    unclamped kernel would write into the guard, inside the allocation) and nothing outside `flat` is read."""
    from phasegen import ops
    from phasegen._lib import PG_STFT_LOGMAG, PG_STFT_REIM
    n_fft, T, B = 256, 40, 4
    hop = n_fft // 4
    P = (T - 1) * hop
    src = torch.randn(B, P, device="cuda") + 3.0
    peak = src.abs().amax(1).contiguous()
    n_dst = 2 * P + 5
    bad = torch.tensor([0, P, n_dst - 10, n_dst + 600, n_dst + 1200], dtype=torch.int64, device="cuda")
    G = 4096                                                # > 1200 + P: every unclamped write lands in the guard
    big = torch.full((n_dst + 2 * G + 1,), -7.0, device="cuda")
    dst = big[G + 1:G + 1 + n_dst]
    ops.peak_normalize_packed(src, peak, bad, dst)
    assert bool((big[:G + 1] == -7.0).all()) and bool((big[G + 1 + n_dst:] == -7.0).all())
    assert torch.equal(dst[:P], src[0] * (1.0 / peak[0])) and torch.equal(dst[P:n_dst - 10], src[1, :P - 5] * (1.0 / peak[1]))
    assert torch.equal(dst[n_dst - 10:], src[2, :10] * (1.0 / peak[2]))
    # peak None: a plain copy
    ops.peak_normalize_packed(src, None, bad, dst)
    assert torch.equal(dst[:P], src[0]) and torch.equal(dst[n_dst - 10:], src[2, :10])
    # the STFT reads inside its view only: NaN all around it, offsets past its end
    n_wave = 2 * P + 5
    buf = torch.full((n_wave + 2 * G,), float("nan"), device="cuda")
    wave = buf[G:G + n_wave]
    wave.copy_(torch.randn(n_wave, device="cuda"))
    frames = torch.full((B,), T, dtype=torch.int32, device="cuda")
    bad_w = torch.tensor([0, P, n_wave - 10, n_wave + 600, n_wave + 1200], dtype=torch.int64, device="cuda")
    a, _ = ops.stft(wave, n_fft, hop, PG_STFT_LOGMAG, want_second=False, clip_frames=frames, clip_offsets=bad_w, frames=T)
    assert bool(torch.isfinite(a).all())
    assert not bool(a[3].any())                             # offsets past the buffer: an empty clip, all zeros
    with pytest.raises(RuntimeError, match="PG_STFT_LOGMAG"):
        ops.stft(wave, n_fft, hop, PG_STFT_REIM, clip_frames=frames, clip_offsets=bad_w, frames=T)


def test_host_buffer_packed_call_equals_device_call():
    from phasegen import synth
    from phasegen.pipeline import PhaseGenPipeline, packed_sub_batches
    n_fft, T, B = 256, 64, 7
    hop = n_fft // 4
    N = (T - 1) * hop
    pipe = PhaseGenPipeline(_net(n_fft, 171), n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)

    def batch(seed):
        rng = np.random.default_rng(seed)
        lengths = [int(v) for v in rng.integers(15 * hop + 1, N + 1, B)]
        lengths[0] |= 1
        w = synth.synthetic_waves(B, N, sr=16000, seed=seed)
        return lengths, torch.cat([w[b, :n] for b, n in enumerate(lengths)]).pin_memory()

    def device_ref(flat, lengths, chunks):
        return torch.cat([pipe.packed(flat[s0:s1].cuda(), lengths[c0:c1], frames=T).cpu()
                          for c0, c1, s0, s1, _ in packed_sub_batches(lengths, chunks)])

    lengths, h_in = batch(172)
    for chunks in (3, [1, 4, 2], pipe.suggest_chunks(B, N, "cuda")):
        h_out = torch.empty_like(h_in).pin_memory()
        assert pipe.run_host_packed(h_in, lengths, h_out, chunks=chunks, frames=T) is h_out
        torch.cuda.synchronize()
        assert torch.equal(h_out, device_ref(h_in, lengths, chunks)), chunks
    # stream of batches: different lengths per call, the same frames, alternating output buffers, six calls back to back
    batches = [batch(180 + i) for i in range(3)]
    want = [device_ref(x, n, [3, 3, 1]) for n, x in batches]
    torch.cuda.synchronize()
    cap = max(x.numel() for _, x in batches)
    outs = [torch.empty(cap).pin_memory() for _ in range(2)]
    pend, got = [None, None], []
    for i in range(6):
        k = i & 1
        if pend[k] is not None:
            pend[k][0].synchronize()
            got.append((pend[k][1], outs[k][:want[pend[k][1]].numel()].clone()))
        n, x = batches[i % 3]
        pend[k] = (pipe.run_host_packed(x, n, outs[k][:x.numel()], chunks=[3, 3, 1], frames=T, pipelined=True), i % 3)
    for k in (0, 1):
        pend[k][0].synchronize()
        got.append((pend[k][1], outs[k][:want[pend[k][1]].numel()].clone()))
    assert len(got) == 6
    for j, y in got:
        assert torch.equal(y, want[j])


def test_fp16_fallback_keeps_the_packed_layout():
    """First-layer weights x 1e7 push d1's output out of the fp16 range: the checked packed call raises, or falls back
    and then equals the bf16x3 packed call and the bf16x3 ragged call."""
    from phasegen.pipeline import PhaseGenPipeline
    n_fft, T, B = 256, 40, 3
    hop = n_fft // 4
    N = (T - 1) * hop
    lengths = [30 * hop + 7, N, 15 * hop + 1]
    net = _net(n_fft, 191)
    with torch.no_grad():
        net.model._parts["down"].weight.mul_(1.0e7)
    wave, flat = _padded_and_flat(B, N, lengths, 16000, seed=192)
    strict = PhaseGenPipeline(net, n_fft, hop, precision="f16mix", per_clip=True, phase_only=True)
    with pytest.raises(OverflowError, match="fp16 range"):
        strict.packed(flat, lengths, check_finite=True)
    soft = PhaseGenPipeline(net, n_fft, hop, precision="f16mix", per_clip=True, phase_only=True, fp16_overflow="fallback")
    got = [t.clone() for t in soft.packed(flat, lengths, check_finite=True, return_intermediates=True)]
    ref = PhaseGenPipeline(net, n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    want = [t.clone() for t in ref.packed(flat, lengths, check_finite=True, return_intermediates=True)]
    for g, w in zip(got, want):
        assert torch.equal(g, w)
    ragged = ref(wave, check_finite=True, return_intermediates=True, lengths=lengths)
    _assert_clips_equal(got[0], ragged[0], lengths)
    assert torch.equal(got[1], ragged[1]) and torch.equal(got[2], ragged[2])


def test_each_packed_clip_meets_the_oracle_bounds():
    from phasegen.pipeline import PhaseGenPipeline, ragged_frames
    n_fft, T, B = 256, 64, 6
    hop, C = n_fft // 4, n_fft // 2
    lengths = _lengths(hop, (T - 1) * hop, seed=201)
    offs = _offsets(lengths)
    net = _net(n_fft, 202)
    sd = {k: v.detach().cpu() for k, v in net.model.state_dict().items()}
    pipe = PhaseGenPipeline(net, n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    _, flat = _padded_and_flat(B, (T - 1) * hop, lengths, 16000, seed=203)
    audio, logmag, phase = pipe.packed(flat, lengths, check_finite=True, return_intermediates=True)
    for b, n in enumerate(lengths):
        T_b = ragged_frames(n, hop)
        w = np.zeros((T_b - 1) * hop)
        w[:n] = flat[offs[b]:offs[b + 1]].cpu().numpy()
        lm = np.log1p(np.abs(stft_np.stft(w, n_fft, hop)[1:]))
        out = unet_torch.unet_forward(sd, torch.from_numpy(lm)[None], torch.float64, per_clip_bn=True)[0].numpy()
        ref = stft_np.generate_audio(stft_np.polar_to_complex(lm, out[:C]), 16000, hop, is_stft=True)[:n]
        got = audio[offs[b]:offs[b + 1]].cpu().numpy()
        assert rel_l2(logmag[b, :T_b].cpu().numpy().T, lm) < 1e-4, b
        assert rel_l2(phase[b, :T_b].cpu().numpy().T, out[:C]) < 1e-3, b
        assert rel_l2(got, ref) < 5e-3, b
        assert abs(snr_db(w[:n], got) - snr_db(w[:n], ref)) < 0.1, b
