"""Host logic of TableTennisPipeline.predict_clips: the stack table over several clips, the network passes over it, the clip blocks,
the split over devices and the `devices` argument.  No GPU needed."""
import pytest
import torch

from upliftingtabletennis_b200 import sharding
from upliftingtabletennis_b200.interface import _Detector, clip_blocks, clip_stack_plan, parse_devices

LENGTHS = [3, 60, 1, 0, 17, 50, 2, 4, 33]


@pytest.mark.parametrize('fps', [1, 3])
def test_stack_plan_covers_every_stack_once_within_its_clip(fps):
    first, offs = clip_stack_plan(LENGTHS, fps)
    assert offs[0] == 0 and len(offs) == len(LENGTHS) + 1 and offs[-1] == len(first)
    f0 = 0
    for c, n in enumerate(LENGTHS):
        stacks = first[offs[c]:offs[c + 1]]
        # the same stacks, in the same order, as predict's sliding window over the clip alone (stride 1)
        assert [s - f0 for s in stacks] == list(range(max(n - fps + 1, 0)))
        assert all(f0 <= s and s + fps <= f0 + n for s in stacks)          # no window crosses a clip
        f0 += n


@pytest.mark.parametrize('fps', [1, 3])
def test_passes_are_full_except_the_last(fps):
    first, _ = clip_stack_plan(LENGTHS, fps)
    plan = _Detector._pass_plan(len(first), _Detector.chunk, False)
    assert [s0 for s0, _ in plan] == list(range(0, len(first), _Detector.chunk))
    assert all(ns == _Detector.chunk for _, ns in plan[:-1]) and 0 < plan[-1][1] <= _Detector.chunk
    assert sum(ns for _, ns in plan) == len(first)


def test_clip_blocks_bound_frames_and_cover_clips_in_order():
    for lengths, cap in ((LENGTHS, 64), ([50] * 64, 512), ([600, 10, 20], 512), ([], 512)):
        blocks = clip_blocks(lengths, cap)
        assert [i for a, b in blocks for i in range(a, b)] == list(range(len(lengths)))
        for a, b in blocks:
            assert b > a and (b - a == 1 or sum(lengths[a:b]) <= cap)
        if lengths == [50] * 64:
            assert [b - a for a, b in blocks] == [10] * 6 + [4]


@pytest.mark.parametrize('n,world', [(64, 1), (64, 8), (7, 3), (3, 8), (0, 2)])
def test_device_split_covers_every_clip_once_in_order(n, world):
    blocks = [sharding.shard_range(n, r, world) for r in range(world)]
    assert [i for a, b in blocks for i in range(a, b)] == list(range(n))


def test_devices_argument():
    assert parse_devices([0, 1, 'cuda:1', torch.device('cuda', 0), 0], 2) == [0, 1, 1, 0, 0]
    for bad in (0, 'cuda:0', torch.device('cuda', 0), [], [2], [-1], ['cpu'], [torch.device('cpu')], ['cuda'], ['gpu0'], [1.0], [True],
                [None]):
        with pytest.raises(ValueError):
            parse_devices(bad, 2)
