"""Host side of ragged batches (PhaseGenPipeline(..., lengths=...)): the per-layer valid-row table, the samples -> frames
rule and the input checks.  No GPU needed."""
import pytest
import torch

from oracle import unet_torch


def _net(C=8, **kw):
    import model
    return model.UNetModel(C, 2 * C, **kw)


def test_valid_row_table_matches_oracle_layer_lengths():
    """For every T the U-Net accepts up to 720 frames, the table's rows are the lengths the float64 oracle's layers
    produce (the lengths do not depend on the channel count)."""
    from phasegen.unet import clip_rows_table
    levels = _net()._levels()
    sd = unet_torch.random_state_dict(8, seed=0, dtype=torch.float64)
    Ts = list(range(24, 721, 8))
    table = clip_rows_table(levels, Ts)
    assert len(table) == len(levels) + 2
    for b, T in enumerate(Ts):
        taps = {}
        unet_torch.unet_forward(sd, torch.zeros(1, 8, T, dtype=torch.float64), taps=taps)
        want = [T] + [taps[k].shape[-1] for k in ("y1", "h2", "h3", "y4", "out")]
        assert [row[b] for row in table] == want, T
        # the up convs land on the skip lengths, so the table covers every buffer of the executor
        assert [taps[k].shape[-1] for k in ("g4", "g3", "g2")] == want[3:0:-1]


def test_min_frames_is_derived_from_the_layer_chain():
    from phasegen.unet import clip_rows_table, min_frames
    levels = _net()._levels()
    assert min_frames(levels) == 24
    with pytest.raises(ValueError):
        clip_rows_table(levels, [16])
    with pytest.raises(ValueError):
        clip_rows_table(levels, [28])


@pytest.mark.parametrize("n_fft", [256, 512, 1024, 2048])
def test_samples_to_frames_rule(n_fft):
    """T_b is the smallest multiple of 8 with (T_b - 1)*hop >= n_b."""
    from phasegen.pipeline import ragged_frames
    hop = n_fft // 4
    for T in (24, 32, 40, 696, 1384):
        n = (T - 1) * hop
        assert ragged_frames(n, hop) == T
        assert ragged_frames(n - 1, hop) == T
        assert ragged_frames(n + 1, hop) == T + 8
    for n in range(0, 40 * hop):
        T = ragged_frames(n, hop)
        assert T % 8 == 0 and (T - 1) * hop >= n and (T - 9) * hop < n


def test_ragged_table_rows():
    from phasegen.pipeline import PhaseGenPipeline, ragged_frames
    n_fft, hop = 256, 64
    pipe = PhaseGenPipeline(_net(128), n_fft, hop, precision="bf16x3", per_clip=True)
    N = 63 * hop
    lengths = [N, 15 * hop + 1, 1000, 2000]
    tab = pipe.ragged_table(4, N, lengths)
    assert tab[0] == lengths
    assert tab[1] == [ragged_frames(n, hop) for n in lengths] == [64, 24, 24, 40]
    assert tab[-1] == tab[1]                                   # the last up conv restores the frame count
    assert pipe.ragged_table(2, N, torch.tensor([N, 3000]))[0] == [N, 3000]


def test_invalid_ragged_inputs_raise_value_error():
    from phasegen.pipeline import PhaseGenPipeline
    n_fft, hop = 256, 64
    N = 63 * hop
    pipe = PhaseGenPipeline(_net(128), n_fft, hop, precision="bf16x3", per_clip=True)
    with pytest.raises(ValueError, match="entries"):
        pipe.ragged_table(3, N, [N, N])
    with pytest.raises(ValueError, match=r"\[0, "):
        pipe.ragged_table(2, N, [N, N + 1])
    with pytest.raises(ValueError, match=r"\[0, "):
        pipe.ragged_table(2, N, [N, -1])
    with pytest.raises(ValueError, match="24 frames"):
        pipe.ragged_table(2, N, [N, 15 * hop])                # 16 frames: below the U-Net's minimum
    pipe.ragged_table(2, N, [N, 15 * hop + 1])                 # 24 frames: the shortest clip
    with pytest.raises(ValueError, match="per_clip"):
        PhaseGenPipeline(_net(128), n_fft, hop, precision="bf16x3", per_clip=False).ragged_table(2, N, [N, N])
    with pytest.raises(ValueError, match="fp32_simt"):
        PhaseGenPipeline(_net(128), n_fft, hop, precision="fp32_simt", per_clip=True).ragged_table(2, N, [N, N])
    with pytest.raises(ValueError, match="fp32_simt"):                     # C = 8 resolves to the SIMT path
        PhaseGenPipeline(_net(8), n_fft, hop, per_clip=True).ragged_table(2, N, [N, N])
    with pytest.raises(ValueError, match="fp32_simt"):                     # the executor options' precision counts too
        PhaseGenPipeline(_net(128), n_fft, hop, per_clip=True, executor_kw={"precision": "fp32_simt"}).ragged_table(2, N, [N, N])


def test_buffer_length_must_hold_every_clips_frames():
    """N must be (T - 1)*hop with T % 8 == 0: otherwise a full-length clip needs more frames (T_b = T + 8 when
    1 + N // hop is a multiple of 8) than the executor's buffers have."""
    from phasegen.pipeline import PhaseGenPipeline, ragged_frames
    n_fft, hop = 256, 64
    pipe = PhaseGenPipeline(_net(128), n_fft, hop, precision="bf16x3", per_clip=True)
    N = 63 * hop + 10                                          # fixed path: T = 64, but ragged_frames(N) = 72
    assert pipe.frames(N) == 64 and ragged_frames(N, hop) == 72
    for bad_N in (N, 62 * hop):                                # not a multiple of hop; T = 63 not a multiple of 8
        with pytest.raises(ValueError, match="T % 8"):
            pipe.ragged_table(2, bad_N, [bad_N, 3000])
        with pytest.raises(ValueError, match="T % 8"):
            pipe.ragged_table(2, bad_N, [3000, 3000])
