"""CPU checks of the jointly computed strips of a sharded k-reciprocal prepare: the gallery ranges each rank computes
(rerank_ranges) and the library's size queries for a rank's part of the strips, which need no GPU."""
import pytest

from ieee_b200 import _lib
from ieee_b200.engine import rerank_owned, rerank_ranges, shard_bounds


def _offsets(sizes):
    return [sum(sizes[:r]) for r in range(len(sizes))]


@pytest.mark.parametrize("sizes", [
    [1700],                                   # world = 1
    [850, 850],                               # unaligned
    [567, 567, 566],
    [100, 1600],                              # a slice under 256 rows
    [30, 30, 30, 30, 30, 30, 30, 1490],       # most ranges empty
    [300, 10, 10, 1380],
    [1000, 600, 95, 5],                       # the last slices end past the last multiple of 256
    [0, 1700, 0],                             # empty slices
])
def test_ranges_tile_the_gallery_at_multiples_of_256(sizes):
    G = sum(sizes)
    offsets = _offsets(sizes)
    ranges = rerank_ranges(offsets, G)
    assert len(ranges) == len(sizes)
    assert ranges[0][0] == 0 and ranges[-1][1] == G
    for (a, b), (c, _) in zip(ranges, ranges[1:]):
        assert b == c
    for r, ((a, b), off, n) in enumerate(zip(ranges, offsets, sizes)):
        assert a <= b
        assert a % 256 == 0 or a == G
        if a < b:
            assert off <= a < off + n                  # a non-empty range starts inside its own slice ...
            assert b - (off + n) < 256                 # ... and reaches fewer than 256 rows past it
        assert a - off < 256 or n == 0


def test_ranges_of_shard_bounds_slices():
    G, world = 1700, 8
    ranges = rerank_ranges([shard_bounds(G, world, r)[0] for r in range(world)], G)
    # slices start at 0, 213, 426, 639, 851, 1063, 1275, 1488: 1063 and 1275 round up to the same 1280
    assert ranges == [(0, 256), (256, 512), (512, 768), (768, 1024), (1024, 1280), (1280, 1280), (1280, 1536), (1536, 1700)]


def test_part_size_queries_need_no_gpu():
    lib = _lib.load()
    Q, G, k1 = 300, 1700, 20
    qa, qb = rerank_owned(Q, G, 2, 1)[:2]
    assert lib.ieee_rerank_stream_part_scratch_bytes(Q, G, k1, qa, qb, 1024, 1700, 512) > 512 * 4 * (qb - qa + 2 * 676)
    assert lib.ieee_rerank_stream_part_scratch_bytes(Q, G, k1, 0, 0, 0, 0, 256) > 0          # a rank without columns
    # the width grows with the budget, in multiples of 256, between 256 and the widest segment
    widths = [lib.ieee_rerank_stream_part_width(Q, G, k1, 0, Q, 0, G, b) for b in (0, 1 << 22, 1 << 23, 1 << 40)]
    assert widths[0] == 256 and widths[-1] == 1792 and widths == sorted(widths) and all(w % 256 == 0 for w in widths)
    # a smaller part fits a wider strip in the same budget
    assert lib.ieee_rerank_stream_part_width(Q, G, k1, 0, 150, 0, 768, 1 << 22) > widths[1]


@pytest.mark.parametrize("args, text", [
    ((300, 1700, 20, 0, 301, 0, 1700, 256), b"query part"),
    ((300, 1700, 20, 200, 100, 0, 1700, 256), b"query part"),
    ((300, 1700, 20, 0, 300, 100, 1700, 256), b"multiple of 256"),
    ((300, 1700, 20, 0, 300, 0, 1800, 256), b"multiple of 256"),
    ((300, 1700, 20, 0, 300, 0, 1700, 300), b"strip width"),
    ((300, 1700, 20, 0, 300, 0, 1700, 0), b"strip width"),
    ((300, 1700, 600, 0, 300, 0, 1700, 256), b"k1"),
])
def test_part_scratch_query_out_of_range(args, text):
    lib = _lib.load()
    assert lib.ieee_rerank_stream_part_scratch_bytes(*args) == 0
    assert text in lib.ieee_last_error()
    if args[-1] == 256:
        assert lib.ieee_rerank_stream_part_width(*args[:-1], 1 << 20) == 0
