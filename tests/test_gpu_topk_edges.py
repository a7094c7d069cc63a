"""GPU parity of the junk-masked top-k (ieee_topk) off its common path: the streaming path for k > 120 on long rows,
each fall-back of the fast path forced by construction, rows that start at every 4-byte offset, and a global index
offset.  Indices and values must equal the CPU oracle's bit for bit."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from ieee_b200 import _lib
from ieee_b200.metrics.rank import topk_ranked_list

pytestmark = pytest.mark.gpu

THREADS = 256          # threads per query row in topk_kernel: thread t's share is the 16-byte vectors i with i % 256 == t


def fast_bound_rank(k):
    """m in topk_select_path: the bound is the m-th smallest of the 256 share leaders (0-based)."""
    return min(2 * k + 8, THREADS) - 1


def assert_topk(got_idx, got_val, d, qp, gp, qc, gc, k, g_offset=0):
    idx_o, val_o = R.topk_kept(d, qp, gp, qc, gc, k)
    idx_o = np.where(idx_o >= 0, idx_o + g_offset, -1)
    idx, val = got_idx.cpu().numpy(), got_val.cpu().numpy()
    assert np.array_equal(idx, idx_o), f"first differing row {np.nonzero((idx != idx_o).any(1))[0][:5]}"
    assert np.array_equal(val.view(np.uint32), val_o.astype(np.float32).view(np.uint32))


def check(d, qp, gp, qc, gc, k):
    """Masked list against the oracle; unmasked list against the oracle and a stable argsort prefix."""
    idx, val = topk_ranked_list(d, qp, gp, qc, gc, k=k)
    assert_topk(idx, val, d, qp, gp, qc, gc, k)
    no_q = np.full(len(qp), -1, dtype=np.int64)                     # a pid no gallery item has: nothing is junk
    idx_u, val_u = topk_ranked_list(d, k=k)
    assert_topk(idx_u, val_u, d, no_q, gp, no_q, gc, k)
    G = d.shape[1]
    want = np.full((d.shape[0], k), -1, dtype=np.int64)
    want[:, :min(k, G)] = np.argsort(d, axis=1, kind="stable")[:, :k]
    assert np.array_equal(idx_u.cpu().numpy(), want)


def special_rows(G, seed):
    """Six rows: continuous values, heavy ties, ties with NaN / +-inf / -0, all equal, almost all inf / NaN, and a row
    whose query finds about half the gallery junk (labels below)."""
    rng = np.random.RandomState(seed)
    d = np.empty((6, G), dtype=np.float32)
    d[0] = rng.rand(G)
    d[1] = rng.randint(0, 8, G)
    d[2] = rng.randint(0, 8, G)
    d[2, 1::3] = -0.0
    d[2, ::3] = 0.0
    d[2, 3::5] = np.inf
    d[2, 2::11] = -np.inf
    d[2, ::7] = np.nan
    d[3] = 1.0
    d[4] = np.where(rng.rand(G) < 0.5, np.inf, np.nan)
    few = rng.choice(G, size=min(G, 5), replace=False)
    d[4, few] = rng.randint(0, 3, few.size)
    d[5] = np.round(rng.rand(G) * 50) / 50
    return d


def special_labels(G, seed):
    rng = np.random.RandomState(seed + 1)
    gp, gc = rng.randint(0, 4, G).astype(np.int64), rng.randint(0, 2, G).astype(np.int64)
    half = rng.rand(G) < 0.5
    gp[half], gc[half] = 9, 9
    qp, qc = rng.randint(0, 4, 6).astype(np.int64), rng.randint(0, 2, 6).astype(np.int64)
    qp[5], qc[5] = 9, 9
    return qp, gp, qc, gc


@pytest.mark.parametrize("G", [7, 1023, 1024, 1025, 4097, 70001])
@pytest.mark.parametrize("k", [121, 128, 129, 500, 1023, 1024])
def test_streaming_path(k, G):
    """k > 120 always streams: threshold filter, compaction of the 2048-entry buffer whenever a tile could overflow
    it.  G <= k (and the half-junk row at G = 1025) leave fewer kept items than k: -1 / inf padding."""
    d = special_rows(G, seed=k * 7 + G)
    check(d, *special_labels(G, seed=k + G), k)


@pytest.fixture(params=[1, 20, 120])
def fast_k(request):
    return request.param


def share_of(G):
    """Share (thread) of every element of a 16-byte-aligned row whose length is a multiple of 4."""
    return (np.arange(G) // 4) % THREADS


def test_fast_path_bound_spent_on_junk(fast_k):
    """Every share's smallest element is junk and these 256 are the row's smallest: the bound (the m-th smallest
    leader) lies among junk items, so no kept element falls under it and n = 0 < k -> general path."""
    k, G = fast_k, 8192
    rng = np.random.RandomState(k)
    d = (1 + rng.rand(4, G)).astype(np.float32)
    lead = np.arange(THREADS) * 4                         # element 4t opens share t's first vector
    d[:, lead] = rng.randint(0, 4, (4, THREADS)) * 0.125
    gp, gc = rng.randint(0, 6, G).astype(np.int64), rng.randint(0, 3, G).astype(np.int64)
    gp[lead], gc[lead] = 7, 1
    qp, qc = np.full(4, 7, dtype=np.int64), np.full(4, 1, dtype=np.int64)
    assert (share_of(G)[lead] == np.arange(THREADS)).all() and THREADS > k + 8
    check(d, qp, gp, qc, gc, k)


def test_fast_path_missing_leaders(fast_k):
    """Only 2k + 4 entries are finite (the rest +inf or NaN, which never lead): fewer than m + 1 = 2k + 8 shares have a
    leader, so no leader has rank m and the bound stays unset -> general path."""
    k, G = fast_k, 8192
    rng = np.random.RandomState(100 + k)
    d = np.where(rng.rand(4, G) < 0.5, np.inf, np.nan).astype(np.float32)
    for r in range(4):
        pos = rng.choice(G, size=2 * k + 4, replace=False)
        d[r, pos] = rng.randint(0, 4, pos.size)
    d[1, rng.choice(G)] = -np.inf
    assert (np.isfinite(d) | np.isneginf(d)).sum(1).max() < fast_bound_rank(k) + 1
    gp, gc = rng.randint(0, 3, G).astype(np.int64), rng.randint(0, 2, G).astype(np.int64)
    qp, qc = rng.randint(0, 3, 4).astype(np.int64), rng.randint(0, 2, 4).astype(np.int64)
    check(d, qp, gp, qc, gc, k)


def test_fast_path_candidate_overflow(fast_k):
    """Shares 0 .. m-1 hold nothing but 0.0 (G / 256 elements each), every other element is in [1, 2): the m smallest
    leaders are zeros, the bound is the smallest leader of the other shares, and every zero -- 256 m > 2048 of them
    (m >= 9), none junk -- falls under it: the candidate buffer overflows -> general path."""
    k, G = fast_k, 65536
    m = fast_bound_rank(k)
    rng = np.random.RandomState(200 + k)
    d = (1 + rng.rand(3, G)).astype(np.float32)
    zero = share_of(G) < m
    d[:, zero] = 0.0
    assert zero.sum() == G // THREADS * m > 2048
    gp, gc = rng.randint(0, 3, G).astype(np.int64), rng.randint(0, 2, G).astype(np.int64)
    gp[zero] = 100                                        # no query has pid 100: the zeros are all kept
    qp, qc = rng.randint(0, 3, 3).astype(np.int64), rng.randint(0, 2, 3).astype(np.int64)
    check(d, qp, gp, qc, gc, k)


@pytest.mark.parametrize("k", [20, 500])
@pytest.mark.parametrize("j", [1, 2, 3])
def test_unaligned_rows(j, k):
    """Rows of a view padded[:, j:j + G] with an odd pitch: row 0 starts 4 j bytes past a 16-byte boundary, so its
    scalar head is 4 - j elements, and later rows take every head in turn.  k = 20: fast path; k = 500: streaming."""
    G, Q, ld = 4097, 6, 4103
    d = special_rows(G, seed=10 * j + k)
    qp, gp, qc, gc = special_labels(G, seed=j)
    padded = torch.full((Q, ld), np.nan, device="cuda")
    view = padded[:, j:j + G]
    view.copy_(torch.from_numpy(d))
    assert view.data_ptr() % 16 == 4 * j and view.stride(0) == ld
    lab = [torch.from_numpy(x).cuda() for x in (qp, qc, gp, gc)]
    idx = torch.empty((Q, k), dtype=torch.int32, device="cuda")
    val = torch.empty((Q, k), dtype=torch.float32, device="cuda")
    _lib.call("ieee_topk", view.data_ptr(), view.stride(0), Q, G, 0, lab[0].data_ptr(), lab[1].data_ptr(),
              lab[2].data_ptr(), lab[3].data_ptr(), k, idx.data_ptr(), val.data_ptr(), _lib.stream())
    assert_topk(idx, val, d, qp, gp, qc, gc, k)


@pytest.mark.parametrize("k", [20, 200])
def test_global_offset(k):
    """A gallery shard starting at global row 2^30: indices shift by the offset; ties still go to the lower index."""
    G, off = 5000, 1 << 30
    d = special_rows(G, seed=k)
    qp, gp, qc, gc = special_labels(G, seed=k)
    idx, val = topk_ranked_list(d, qp, gp, qc, gc, k=k, g_offset=off)
    assert_topk(idx, val, d, qp, gp, qc, gc, k, g_offset=off)
