"""wf_host_shard_columns: which trace columns each rank of a sharded proof owns (include/winterfell_b200.h). Host code, no GPU."""
import pytest

import winterfell_b200 as wf

WORLDS = [2, 4, 8, 16, 32, 64]


@pytest.mark.parametrize("world", WORLDS)
def test_ranges_cover_the_trace_in_whole_segments(world):
    for width in range(1, 256):
        ranges = [wf.shard_columns(width, world, r) for r in range(world)]
        nxt = 0
        for first, count in ranges:   # contiguous, in rank order, every column exactly once
            assert first == nxt, (width, ranges)
            nxt = first + count
        assert nxt == width, (width, ranges)
        for first, count in ranges:   # boundaries on segment boundaries (the last column ends the trace)
            assert first % 8 == 0 and ((first + count) % 8 == 0 or first + count == width), (width, first, count)
        segs = [(count + 7) // 8 for _, count in ranges]
        assert max(segs) - min(segs) <= 1, (width, segs)
        assert sum(segs) == (width + 7) // 8
        if width % (8 * world) == 0:   # the blocks wf_prove_fib_sharded takes
            assert ranges == [(r * width // world, width // world) for r in range(world)]


def test_narrow_traces_leave_ranks_without_columns():
    # one segment: one rank owns all of it, the others none
    for world in WORLDS:
        counts = [wf.shard_columns(6, world, r)[1] for r in range(world)]
        assert sorted(counts) == [0] * (world - 1) + [6]
    assert [wf.shard_columns(24, 4, r) for r in range(4)] == [(0, 0), (0, 8), (8, 8), (16, 8)]
    assert [wf.shard_columns(12, 2, r) for r in range(2)] == [(0, 8), (8, 4)]


@pytest.mark.parametrize("width,world,rank", [(0, 2, 0), (256, 2, 0), (8, 1, 0), (8, 0, 0), (8, 3, 0), (8, 6, 1), (8, 2, 2),
                                              (8, 2, -1), (8, -2, 0)])
def test_invalid_arguments_are_refused(width, world, rank):
    with pytest.raises(wf.WfError):
        wf.shard_columns(width, world, rank)


def test_null_outputs_are_refused():
    import ctypes as C
    L = wf.lib()
    c = C.c_uint32(0)
    assert L.wf_host_shard_columns(8, 2, 0, None, C.byref(c)) != wf.WF_OK
    assert L.wf_host_shard_columns(8, 2, 0, C.byref(c), None) != wf.WF_OK
