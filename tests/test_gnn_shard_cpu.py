"""CPU checks of GNN re-ranking shared by a query_group: the layout query and the split of rows and queries."""
import ctypes as C

import pytest

from ieee_b200 import _lib
from ieee_b200.engine import rerank_owned


def layout(Q, G, k1, k2, sizes=None):
    off = (C.c_size_t * 10)()
    arg = None if sizes is None else (C.c_int64 * 6)(*sizes)
    rc = _lib.load().ieee_gnn_stream_layout(Q, G, k1, k2, arg, off)
    return rc, list(off)


def test_layout_needs_no_gpu():
    Q, G, k1 = 300, 1700, 26
    N = Q + G
    rc, off = layout(Q, G, k1, 7)
    assert rc == _lib.OK
    counts = off[:4]
    # four int32 [N] count arrays, 256-byte aligned, disjoint, inside the scratch of the graph calls
    assert all(o % 256 == 0 for o in counts) and all(b - a >= 4 * N for a, b in zip(counts, counts[1:]))
    assert counts[3] + 4 * N <= _lib.load().ieee_gnn_stream_scratch_bytes(Q, G, k1, 0)
    nb1, na1, nb2 = 90000, 120000, 150000
    rc, off = layout(Q, G, k1, 7, (0, 0, 0, nb1, na1, nb2))
    assert rc == _lib.OK and off[:4] == counts
    work = off[4:]                 # B1 columns, values; A1 columns, values; B2 columns, values
    assert all(o % 256 == 0 for o in work)
    for (c, v), n in zip(((work[0], work[1]), (work[2], work[3]), (work[4], work[5])), (nb1, na1, nb2)):
        assert v - c >= 4 * n
    assert work[0] < work[1] < work[2] < work[3] < work[4] < work[5]
    assert work[5] - work[4] >= 4 * nb2


def test_layout_rejects_what_the_phases_reject():
    lib = _lib.load()
    assert layout(10, 10, 21, 7)[0] == _lib.ERR_INVALID          # k1 > N
    assert b"exceeds" in lib.ieee_last_error()
    assert layout(100, 1000, 26, 27)[0] == _lib.ERR_INVALID      # k2 > k1
    assert layout(0, 1000, 26, 7)[0] == _lib.ERR_INVALID
    assert layout(1 << 19, (1 << 19) + 1, 26, 7)[0] == _lib.ERR_INVALID


@pytest.mark.parametrize("Q,G", [(300, 1700), (1, 1), (10000, 140000), (100, 70000)])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_query_rows_are_the_owned_queries(Q, G, world):
    """Each rank evaluates the queries whose rows of A it computes: rows [q0, q1) of rerank_owned, which tile [0, Q) in
    rank order; with fewer than 256 queries per rank, the later ranks evaluate none."""
    parts = [rerank_owned(Q, G, world, r)[:2] for r in range(world)]
    assert parts[0][0] == 0 and parts[-1][1] == Q
    assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
    if Q <= 256:
        assert parts[0] == (0, Q) and all(p == (Q, Q) for p in parts[1:])
