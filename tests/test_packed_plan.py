"""Host side of packed clips (PhaseGenPipeline.packed / run_host_packed): lengths -> offsets -> sub-batches, and the input
checks.  No GPU needed."""
import pytest
import torch


def _pipe(C=128):
    import model
    from phasegen.pipeline import PhaseGenPipeline
    return PhaseGenPipeline(model.UNetModel(C, 2 * C), 2 * C, C // 2, precision="bf16x3", per_clip=True)


def test_offsets_are_the_running_sum():
    from phasegen.pipeline import packed_offsets
    assert packed_offsets([5, 3, 7]) == [0, 5, 8, 15]
    assert packed_offsets(torch.tensor([4, 1]).tolist()) == [0, 4, 5]


@pytest.mark.parametrize("chunks,want", [
    (2, [(0, 3), (3, 5)]),                                     # equal sub-batches, the last one shorter
    ([1, 3, 1], [(0, 1), (1, 4), (4, 5)]),                     # explicit unequal sizes
    ([1, 2, 1, 1], [(0, 1), (1, 3), (3, 4), (4, 5)]),          # suggest_chunks-style ramp (head, middles, tail)
    (1, [(0, 5)]),
])
def test_sub_batches_cover_contiguous_sample_ranges(chunks, want):
    from phasegen.pipeline import packed_offsets, packed_sub_batches
    lengths = [1537, 960, 2049, 1001, 3000]                    # odd offsets and offsets that are not multiples of 4
    offs = packed_offsets(lengths)
    subs = packed_sub_batches(lengths, chunks)
    assert [(c0, c1) for c0, c1, _, _, _ in subs] == want
    s_prev = 0
    for c0, c1, s0, s1, rebased in subs:
        assert (s0, s1) == (offs[c0], offs[c1]) and s0 == s_prev
        assert rebased == [o - s0 for o in offs[c0:c1 + 1]] and rebased[0] == 0 and rebased[-1] == s1 - s0
        s_prev = s1
    assert s_prev == sum(lengths)


def test_sub_batch_sizes_must_add_up():
    from phasegen.pipeline import packed_sub_batches
    with pytest.raises(RuntimeError, match="add up"):
        packed_sub_batches([1000, 2000, 3000], [1, 1])
    with pytest.raises(RuntimeError, match="add up"):
        packed_sub_batches([1000, 2000, 3000], [3, 0])


def test_packed_table_equals_the_ragged_table_of_the_padded_call():
    from phasegen.pipeline import ragged_frames
    pipe = _pipe()
    hop = pipe.hop
    lengths = [40 * hop + 3, 15 * hop + 1, 2001, 63 * hop]
    T, table, offs = pipe.packed_table(torch.zeros(sum(lengths)), lengths)
    assert T == ragged_frames(max(lengths), hop) == 64
    assert table == pipe.ragged_table(4, (T - 1) * hop, lengths)
    assert offs == [0, lengths[0], sum(lengths[:2]), sum(lengths[:3]), sum(lengths)]
    T2, table2, _ = pipe.packed_table(torch.zeros(sum(lengths)), lengths, frames=96)   # a larger bucket keeps the clips' tables
    assert T2 == 96 and table2 == table


def test_packed_inputs_raise_value_error():
    pipe = _pipe()
    hop = pipe.hop
    lengths = [40 * hop + 3, 15 * hop + 1]
    n = sum(lengths)
    with pytest.raises(ValueError, match="1-D"):
        pipe.packed_table(torch.zeros(2, n // 2), lengths)
    with pytest.raises(ValueError, match="add up"):
        pipe.packed_table(torch.zeros(n + 1), lengths)
    with pytest.raises(ValueError, match="add up"):
        pipe.packed_table(torch.zeros(n), lengths[:1])
    with pytest.raises(ValueError, match="multiple of 8"):
        pipe.packed_table(torch.zeros(n), lengths, frames=52)
    with pytest.raises(ValueError, match="at least 48"):
        pipe.packed_table(torch.zeros(n), lengths, frames=40)   # the longest clip needs 48 frames
    with pytest.raises(ValueError, match="empty"):
        pipe.packed_table(torch.zeros(0), [])
    # the ragged call's own checks: the U-Net's minimum of 24 frames, negative lengths, per_clip, fp32_simt
    with pytest.raises(ValueError, match="24 frames"):
        pipe.packed_table(torch.zeros(n - 1), [lengths[0], 15 * hop])
    with pytest.raises(ValueError, match=r"\[0, "):
        pipe.packed_table(torch.zeros(n - 2 * lengths[1]), [lengths[0], -lengths[1]])
    import model
    from phasegen.pipeline import PhaseGenPipeline
    for kw, msg in ((dict(precision="bf16x3", per_clip=False), "per_clip"), (dict(precision="fp32_simt"), "fp32_simt")):
        with pytest.raises(ValueError, match=msg):
            PhaseGenPipeline(model.UNetModel(128, 256), 256, 64, **kw).packed_table(torch.zeros(n), lengths, None, kw["precision"])
    # the host form takes the same checks before it touches a device
    with pytest.raises(ValueError, match="add up"):
        pipe.run_host_packed(torch.zeros(n + 1), lengths, torch.zeros(n + 1))
