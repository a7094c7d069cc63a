"""CPU checks of re-ranking over a sharded gallery: how the strips are shared out, and the windowed workspace size."""
import pytest

from ieee_b200 import _lib
from ieee_b200.engine import rerank_owned


@pytest.mark.parametrize("Q,G", [(1, 1), (300, 1700), (836, 836), (256, 512), (20000, 300000), (5, 70000)])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_owned_samples_tile_both_segments(Q, G, world):
    parts = [rerank_owned(Q, G, world, r) for r in range(world)]
    for seg, n in ((0, Q), (2, G)):
        ranges = [(p[seg], p[seg + 1]) for p in parts]
        assert ranges[0][0] == 0 and ranges[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))            # in rank order, no gap, no overlap
        assert all(a <= b and (a % 256 == 0 or a == b == n) for a, b in ranges)     # (an empty share sits at the end)
        strips = [(b - a + 255) // 256 for a, b in ranges]
        assert max(strips) - min(strips) <= 1


def test_window_workspace_size():
    """Needs no GPU; the full window is the one-GPU size, and the size shrinks with the window."""
    lib = _lib.load()
    Q, G = 20000, 300000
    full = lib.ieee_rerank_stream_workspace_bytes(Q, G, 20, 6)
    assert lib.ieee_rerank_stream_window_workspace_bytes(Q, G, 20, 6, G) == full > 0
    sizes = [lib.ieee_rerank_stream_window_workspace_bytes(Q, G, 20, 6, gs) for gs in (G, G // 2, G // 8, 1, 0)]
    assert all(a > b > 0 for a, b in zip(sizes, sizes[1:]))
    # V of all N rows stays; the expansion and the index (8 bytes per entry each) shrink with the window: k2 (k1 + 1)
    # (round(k1 / 2) + 2) entries and a count, about 24 KB, per window row at k1 = 20, k2 = 6
    per_row = (sizes[0] - sizes[1]) / (G - G // 2)
    assert abs(per_row - (16 * 6 * 21 * 12 + 4)) < 1
    assert lib.ieee_rerank_stream_window_workspace_bytes(Q, G, 20, 1, G) == lib.ieee_rerank_stream_workspace_bytes(Q, G, 20, 1)
    assert lib.ieee_rerank_stream_window_workspace_bytes(Q, G, 20, 6, G + 1) == 0
    assert b"window" in lib.ieee_last_error()
    assert lib.ieee_rerank_stream_window_workspace_bytes(Q, G, 20, 22, G) == 0          # k2 > k1 + 1


def test_v_layout_needs_no_gpu():
    import ctypes as C
    lib = _lib.load()
    cap, oc, ov, on = C.c_int64(), C.c_size_t(), C.c_size_t(), C.c_size_t()
    assert lib.ieee_rerank_stream_v_layout(300, 1700, 20, 6, C.byref(cap), C.byref(oc), C.byref(ov), C.byref(on)) == _lib.OK
    assert cap.value == 21 * 12                                  # (k1 + 1) (round(k1 / 2) + 2)
    assert oc.value < ov.value < on.value and ov.value - oc.value >= 2000 * cap.value * 4 and oc.value % 256 == 0
    assert on.value + 2000 * 4 <= lib.ieee_rerank_stream_window_workspace_bytes(300, 1700, 20, 6, 0)
    assert lib.ieee_rerank_stream_v_layout(5, 10, 20, 6, C.byref(cap), C.byref(oc), C.byref(ov), C.byref(on)) != _lib.OK
