"""Ragged batches on the GPU: clips of different lengths in one PhaseGenPipeline call, each equal to running that clip
alone, zero-padded to its own frame count (pipeline.ragged_frames)."""
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
    """Six seeded lengths: the full buffer, the shortest clip (24 frames), one not a multiple of hop, and a pair whose
    frame counts differ by exactly 8."""
    from phasegen.pipeline import ragged_frames
    rng = np.random.default_rng(seed)
    n_min = 15 * hop + 1
    a = int(rng.integers(40 * hop, N - 16 * hop))
    n = [N, n_min, int(rng.integers(n_min, N)) // hop * hop + int(rng.integers(1, hop)), a, a - 8 * hop, int(rng.integers(n_min, N))]
    assert ragged_frames(n[3], hop) - ragged_frames(n[4], hop) == 8 and n[2] % hop
    return n


def _ragged_wave(B, N, lengths, sr, seed):
    from phasegen import synth
    wave = synth.synthetic_waves(B, N, sr=sr, seed=seed, device="cuda")
    for b, n in enumerate(lengths):
        wave[b, n:] = float("nan")                          # never read
    return wave


def _alone(pipe, wave, b, n, hop):
    """The fixed-shape pipeline on clip b alone, zero-padded to (T_b - 1)*hop samples."""
    from phasegen.pipeline import ragged_frames
    x = torch.zeros(1, (ragged_frames(n, hop) - 1) * hop, device="cuda")
    x[0, :n] = wave[b, :n]
    audio, lm, ph = pipe(x, return_intermediates=True)
    return x[0].cpu().numpy().astype(np.float64), audio[0].cpu().numpy(), lm[0].cpu().numpy(), ph[0].cpu().numpy()


def _check_tail_zero(audio, logmag, phase, lengths, hop):
    from phasegen.pipeline import ragged_frames
    assert bool(torch.isfinite(audio).all() and torch.isfinite(logmag).all() and torch.isfinite(phase).all())
    for b, n in enumerate(lengths):
        T_b = ragged_frames(n, hop)
        assert not bool(audio[b, n:].any()) and not bool(logmag[b, T_b:].any()) and not bool(phase[b, T_b:].any()), b


@pytest.mark.parametrize("prec", ["bf16x3", "f16mix1"])
@pytest.mark.parametrize("n_fft,T,B", [(256, 40, 3), (1024, 696, 48)])
def test_full_lengths_are_bit_identical_to_the_fixed_call(n_fft, T, B, prec):
    from phasegen import synth
    from phasegen.pipeline import PhaseGenPipeline
    hop = n_fft // 4
    N = (T - 1) * hop
    pipe = PhaseGenPipeline(_net(n_fft, 61), n_fft, hop, precision=prec, per_clip=True, phase_only=True)
    wave = synth.synthetic_waves(B, N, sr=44100, seed=62, device="cuda")
    fixed = [t.clone() for t in pipe(wave, return_intermediates=True)]
    ragged = pipe(wave, return_intermediates=True, lengths=[N] * B)
    for f, r in zip(fixed, ragged):
        assert torch.equal(f, r)


@pytest.mark.parametrize("n_fft", [256, 512])
def test_each_clip_equals_the_standalone_call(n_fft):
    from phasegen.pipeline import PhaseGenPipeline, ragged_frames
    hop, T, B = n_fft // 4, 64, 6
    N = (T - 1) * hop
    lengths = _lengths(hop, N, seed=n_fft)
    pipe = PhaseGenPipeline(_net(n_fft, 71), n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    wave = _ragged_wave(B, N, lengths, 16000, seed=72)
    audio, logmag, phase = [t.clone() for t in pipe(wave, check_finite=True, return_intermediates=True, lengths=lengths)]
    assert pipe.nonfinite_clips(B) == []
    _check_tail_zero(audio, logmag, phase, lengths, hop)
    for b, n in enumerate(lengths):
        T_b = ragged_frames(n, hop)
        _, a1, lm1, ph1 = _alone(pipe, wave, b, n, hop)
        assert rel_l2(audio[b, :n].cpu().numpy(), a1[:n]) <= 1e-4, b
        assert rel_l2(logmag[b, :T_b].cpu().numpy(), lm1) <= 1e-4, b
        assert rel_l2(phase[b, :T_b].cpu().numpy(), ph1) <= 1e-4, b


@pytest.mark.parametrize("n_fft", [256, 512])
def test_each_clip_meets_the_oracle_bounds(n_fft):
    from phasegen.pipeline import PhaseGenPipeline, ragged_frames
    hop, T, B = n_fft // 4, 64, 6
    C = n_fft // 2
    N = (T - 1) * hop
    lengths = _lengths(hop, N, seed=n_fft + 1)
    net = _net(n_fft, 81)
    sd = {k: v.detach().cpu() for k, v in net.model.state_dict().items()}
    pipe = PhaseGenPipeline(net, n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    wave = _ragged_wave(B, N, lengths, 16000, seed=82)
    audio, logmag, phase = pipe(wave, check_finite=True, return_intermediates=True, lengths=lengths)
    for b, n in enumerate(lengths):
        T_b = ragged_frames(n, hop)
        w = np.zeros((T_b - 1) * hop)
        w[:n] = wave[b, :n].cpu().numpy()
        lm = np.log1p(np.abs(stft_np.stft(w, n_fft, hop)[1:]))
        out = unet_torch.unet_forward(sd, torch.from_numpy(lm)[None], torch.float64, per_clip_bn=True)[0].numpy()
        ref = stft_np.generate_audio(stft_np.polar_to_complex(lm, out[:C]), 16000, hop, is_stft=True)[:n]
        got = audio[b, :n].cpu().numpy()
        assert rel_l2(logmag[b, :T_b].cpu().numpy().T, lm) < 1e-4, b
        assert rel_l2(phase[b, :T_b].cpu().numpy().T, out[:C]) < 1e-3, b
        assert rel_l2(got, ref) < 5e-3, b
        assert abs(snr_db(w[:n], got) - snr_db(w[:n], ref)) < 0.1, b


def test_stale_rows_of_a_longer_call_are_cleared():
    from phasegen import synth
    from phasegen.pipeline import PhaseGenPipeline
    n_fft, T, B = 256, 64, 6
    hop = n_fft // 4
    N = (T - 1) * hop
    lengths = _lengths(hop, N, seed=91)
    net = _net(n_fft, 92)
    pipe = PhaseGenPipeline(net, n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    pipe(synth.synthetic_waves(B, N, sr=16000, seed=93, device="cuda"))        # full-length rows everywhere
    wave = _ragged_wave(B, N, lengths, 16000, seed=94)
    got = [t.clone() for t in pipe(wave, return_intermediates=True, lengths=lengths)]
    fresh = PhaseGenPipeline(_net(n_fft, 92), n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)   # same weights, own executors
    want = fresh(wave, return_intermediates=True, lengths=lengths)
    for g, w in zip(got, want):
        assert torch.equal(g, w)
    ex = pipe._executors[-1]
    table = pipe.ragged_table(B, N, lengths)
    bufs = [(ex.x0, table[1])] + [(op, table[i + 2]) for i in range(ex.D) for op in (ex.a[i], ex.cat[i]) if op is not None]
    for op, rows in bufs:
        for plane in (op.hi, op.lo):
            if plane is None:
                continue
            for b, L_b in enumerate(rows):
                assert not bool(plane[b, L_b:].any()), (op.L, b, L_b)


def test_full_size_ragged_batch():
    """BASELINE shape (C 512, T 696), bench precision, 48 clips of 1 s to 4 s at 44.1 kHz: whole-clip norm tiles, merged
    tiles and CTA pairs with per-clip lengths."""
    from phasegen.pipeline import PhaseGenPipeline, ragged_frames
    n_fft, T, B, sr = 1024, 696, 48, 44100
    hop, C = n_fft // 4, n_fft // 2
    N = (T - 1) * hop
    rng = np.random.default_rng(101)
    lengths = [int(v) for v in rng.integers(sr, 4 * sr + 1, B)]
    net = _net(n_fft, 102)
    pipe = PhaseGenPipeline(net, n_fft, hop, precision="f16mix1", per_clip=True, phase_only=True)
    wave = _ragged_wave(B, N, lengths, sr, seed=103)
    audio, logmag, phase = [t.clone() for t in pipe(wave, check_finite=True, return_intermediates=True, lengths=lengths)]
    _check_tail_zero(audio, logmag, phase, lengths, hop)
    for b in (0, 17, 40):
        n = lengths[b]
        _, a1, _, _ = _alone(pipe, wave, b, n, hop)
        assert rel_l2(audio[b, :n].cpu().numpy(), a1[:n]) <= 1e-4, b
    b = int(np.argmin(lengths))
    n, T_b = lengths[b], ragged_frames(lengths[b], hop)
    sd = {k: v.detach().cpu() for k, v in net.model.state_dict().items()}
    w = np.zeros((T_b - 1) * hop)
    w[:n] = wave[b, :n].cpu().numpy()
    lm = np.log1p(np.abs(stft_np.stft(w, n_fft, hop)[1:]))
    out = unet_torch.unet_forward(sd, torch.from_numpy(lm)[None], torch.float64, per_clip_bn=True)[0].numpy()
    assert rel_l2(phase[b, :T_b].cpu().numpy().T, out[:C]) <= 1e-3


def test_fp16_fallback_keeps_the_lengths():
    """First-layer weights x 1e7 push d1's output out of the fp16 range: the checked ragged call raises, or falls back
    and then equals the bf16x3 ragged call."""
    from phasegen import synth
    from phasegen.pipeline import PhaseGenPipeline
    n_fft, T, B = 256, 40, 3
    hop = n_fft // 4
    N = (T - 1) * hop
    lengths = [N, 15 * hop + 1, 30 * hop + 7]
    net = _net(n_fft, 111)
    with torch.no_grad():
        net.model._parts["down"].weight.mul_(1.0e7)
    wave = _ragged_wave(B, N, lengths, 16000, seed=112)
    strict = PhaseGenPipeline(net, n_fft, hop, precision="f16mix", per_clip=True, phase_only=True)
    with pytest.raises(OverflowError, match="fp16 range"):
        strict(wave, check_finite=True, lengths=lengths)
    soft = PhaseGenPipeline(net, n_fft, hop, precision="f16mix", per_clip=True, phase_only=True, fp16_overflow="fallback")
    got = [t.clone() for t in soft(wave, check_finite=True, return_intermediates=True, lengths=lengths)]
    ref = PhaseGenPipeline(net, n_fft, hop, precision="bf16x3", per_clip=True, phase_only=True)
    want = ref(wave, check_finite=True, return_intermediates=True, lengths=lengths)
    for g, w in zip(got, want):
        assert torch.equal(g, w)
    _check_tail_zero(*got, lengths, hop)


def test_ragged_call_rejects_bad_lengths():
    from phasegen.pipeline import PhaseGenPipeline
    n_fft, T, B = 256, 40, 2
    hop = n_fft // 4
    N = (T - 1) * hop
    wave = torch.zeros(B, N, device="cuda")
    pipe = PhaseGenPipeline(_net(n_fft, 121), n_fft, hop, precision="bf16x3", per_clip=True)
    for bad in ([N], [N, N + 1], [N, 15 * hop]):
        with pytest.raises(ValueError):
            pipe(wave, lengths=bad)
    with pytest.raises(ValueError, match="T % 8"):            # 1 + N // hop = 40 frames, but n_b = N needs 48
        pipe(torch.zeros(B, N + 10, device="cuda"), lengths=[N + 10, N])
    for kw in (dict(precision="fp32_simt", per_clip=True), dict(precision="bf16x3", per_clip=False)):
        with pytest.raises(ValueError):
            PhaseGenPipeline(pipe.model, n_fft, hop, **kw)(wave, lengths=[N, N])
