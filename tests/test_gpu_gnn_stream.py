"""Streamed GNN re-ranking inside RetrievalEvaluator (rerank="gnn"): neighbours, S and the sparse adjacency have the
bits of the dense path (ieee_gnn_rerank on the NEG_DOT contraction of X_u), the final product stays within 1e-6 of an
fp64 product, every strip width and block size gives the same bits, and a set past both dense limits runs."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from ieee_b200 import _lib
from ieee_b200.engine import RetrievalEvaluator
from ieee_b200.metrics.distance import _device_distmat
from ieee_b200.metrics.rank import evaluate_device, topk_ranked_list
from ieee_b200.testing import make_retrieval_set, market1501_shaped, rgbnt201_shaped
from ieee_b200.utils.gnn_reranking import gnn_reranking_distmat

gpu = pytest.mark.gpu
r32 = lambda x: (x + 31) // 32 * 32


def strip_budget(N, k1, rows):
    """block_bytes that gives strips of `rows` rows: the library sizes a strip row at 4 * (N rounded up to 32 + k1) bytes."""
    return rows * 4 * (r32(N) + k1)


def unit(t):
    return torch.nn.functional.normalize(t.float(), dim=1)


def dense_gnn(qf, gf, k1, k2):
    """rank, S and A of the dense path (ieee_gnn_rerank on -(X_u X_u^T)), and its -(A_q A_g^T)."""
    Q = qf.shape[0]
    xu = torch.cat((qf, gf))
    N = xu.shape[0]
    neg = torch.empty((N, r32(N)), dtype=torch.float32, device="cuda")[:, :N]
    _device_distmat(xu, xu, "neg_dot", out=neg)
    rank = torch.empty((N, k1), dtype=torch.int32, device="cuda")
    val = torch.empty((N, k1), dtype=torch.float32, device="cuda")
    _lib.call("ieee_topk", neg.data_ptr(), neg.stride(0), N, N, 0, None, None, None, None, k1, rank.data_ptr(), val.data_ptr(),
              _lib.stream())
    A = torch.empty((N, r32(N)), dtype=torch.float32, device="cuda")
    ws = torch.empty(_lib.load().ieee_gnn_rerank_workspace_bytes(N, k1), dtype=torch.uint8, device="cuda")
    _lib.call("ieee_gnn_rerank", neg.data_ptr(), neg.stride(0), N, k1, k2, A.data_ptr(), A.stride(0), ws.data_ptr(), ws.numel(),
              _lib.stream())
    del neg
    A = A[:, :N]
    return rank, val * val, A, _device_distmat(A[:Q], A[Q:], "neg_dot")


def densify(rr, N):
    ptr = rr["a_ptr"]
    rows = torch.repeat_interleave(torch.arange(N, device="cuda"), ptr.diff())
    A = torch.zeros((N, N), dtype=torch.float32, device="cuda")
    A[rows, rr["a_col"].long()] = rr["a_val"]
    return A, rows


def check_layout(rr, N, Q, A):
    """CSR columns ascending per row; the CSC holds exactly the gallery rows of A, rows ascending per column."""
    A_s, rows = densify(rr, N)
    col = rr["a_col"].long()
    same_row = rows[1:] == rows[:-1]
    assert bool((col[1:][same_row] > col[:-1][same_row]).all())
    gp = rr["g_ptr"]
    assert gp[0].item() == 0 and gp[-1].item() == rr["g_row"].numel() == (rr["a_ptr"][N] - rr["a_ptr"][Q]).item()
    gcols = torch.repeat_interleave(torch.arange(N, device="cuda"), gp.diff())
    g = rr["g_row"].long()
    same_col = gcols[1:] == gcols[:-1]
    assert bool((g[1:][same_col] > g[:-1][same_col]).all())
    Ag = torch.zeros((N - Q, N), dtype=torch.float32, device="cuda")
    Ag[g, gcols] = rr["g_val"]
    assert torch.equal(Ag, A[Q:])
    return A_s


def check_against_dense(s, k1=26, k2=7, dtype=torch.float32, block_bytes=None, max_rank=20):
    qf, gf = unit(s.qf).cuda().to(dtype), unit(s.gf).cuda().to(dtype)
    Q, G = qf.shape[0], gf.shape[0]
    N = Q + G
    kw = {} if block_bytes is None else {"block_bytes": block_bytes}
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, max_rank=max_rank, rerank="gnn", k1=k1, k2=k2, **kw)
    cmc, mAP, info = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    rr = ev._rr
    rank, S, A, out_d = dense_gnn(qf, gf, k1, k2)
    if dtype == torch.float32:
        assert torch.equal(out_d, gnn_reranking_distmat(qf, gf, k1, k2))
    assert torch.equal(rr["rank"], rank) and torch.equal(rr["S"], S)
    A_s = check_layout(rr, N, Q, A)
    assert torch.equal(A_s, A)
    out = info["distmat"]
    if k2 == 1:
        assert torch.equal(out, out_d)
    else:
        ref = -(A[:Q].double() @ A[Q:].double().T)
        err_s, err_d = (out.double() - ref).abs().max().item(), (out_d.double() - ref).abs().max().item()
        print("max |d| vs fp64: sparse %.3g dense %.3g" % (err_s, err_d))
        assert err_s <= 1e-6 and err_s <= err_d + 1e-6, (err_s, err_d)
    cmc_d, summary, st = evaluate_device(out, s.q_pids, s.g_pids, s.q_camids, s.g_camids, max_rank)
    assert np.array_equal(cmc, cmc_d.cpu().numpy())
    assert mAP == float(summary.mAP) and info["mINP"] == float(summary.mINP)
    assert torch.equal(info["ap"], st.ap) and torch.equal(info["first"], st.first)
    return ev, qf, info


@gpu
def test_c3_shape_self_duplicates():
    """Query set == gallery set: exact duplicates, ties and hubs."""
    check_against_dense(rgbnt201_shaped())


@gpu
def test_market_shaped():
    s = market1501_shaped()
    ev, qf, info = check_against_dense(s)
    idx, val = ev.ranked_lists(qf, s.q_pids, s.q_camids, k=10)
    idx_d, val_d = topk_ranked_list(info["distmat"], s.q_pids, s.g_pids, s.q_camids, s.g_camids, k=10)
    assert torch.equal(idx.cpu(), torch.as_tensor(idx_d).cpu()) and torch.equal(val.cpu(), torch.as_tensor(val_d).cpu())


@gpu
@pytest.mark.parametrize("Q,G,k1,k2", [(5, 16, 21, 6), (8, 13, 20, 20), (1, 30, 30, 3), (30, 1, 30, 7), (6, 10, 15, 1)])
def test_tiny_shapes_k1_near_n(Q, G, k1, k2):
    s = make_retrieval_set(Q, G, 4, 2, dim=48, sigma=1.5, seed=Q * 100 + G)
    s.q_pids, s.g_pids = np.arange(Q, dtype=np.int64) % 2, np.arange(G, dtype=np.int64) % 2
    s.q_camids, s.g_camids = np.zeros(Q, dtype=np.int64), np.ones(G, dtype=np.int64)
    check_against_dense(s, k1=k1, k2=k2, max_rank=min(5, G))


@gpu
@pytest.mark.parametrize("k1,k2", [(26, 7), (20, 6), (10, 1), (12, 12)])
def test_parameters(k1, k2):
    s = make_retrieval_set(420, 1900, 40, 4, dim=256, sigma=2.5, seed=k1 + k2)
    check_against_dense(s, k1=k1, k2=k2)


@gpu
def test_bf16():
    s = make_retrieval_set(300, 1700, 30, 4, dim=384, sigma=2.5, seed=22)
    ev, _, _ = check_against_dense(s, dtype=torch.bfloat16)
    assert ev.precision == "bf16"


@gpu
def test_normalize_feature_within_tolerance():
    """normalize_feature=True normalises while packing, not as torch does: compared with a tolerance only."""
    s = make_retrieval_set(300, 1700, 30, 4, dim=256, sigma=2.5, seed=5)
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, normalize_feature=True, rerank="gnn")
    cmc, mAP, info = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True)
    ref = gnn_reranking_distmat(unit(s.qf).cuda(), unit(s.gf).cuda(), 26, 7)
    close = (info["distmat"] - ref).abs() <= 1e-5
    assert close.float().mean().item() > 0.99
    cmc_r, summary, _ = evaluate_device(ref, s.q_pids, s.g_pids, s.q_camids, s.g_camids, 20)
    assert abs(mAP - float(summary.mAP)) < 1e-3


@gpu
def test_cpu_restatement():
    """Within 1e-5 of the oracle's gnn_reranking, as test_gnn_reranking_matches_restatement allows the dense path."""
    s = make_retrieval_set(60, 300, 12, 3, dim=256, sigma=1.5, seed=26)
    xq, xg = unit(s.qf), unit(s.gf)
    for k1, k2 in ((26, 7), (10, 1)):
        ev = RetrievalEvaluator(xg.cuda(), s.g_pids, s.g_camids, rerank="gnn", k1=k1, k2=k2)
        _, _, info = ev.evaluate(xq.cuda(), s.q_pids, s.q_camids, return_distmat=True)
        cos_o = R.gnn_reranking(xq.numpy(), xg.numpy(), k1, k2, return_similarity=True)
        assert np.abs(-info["distmat"].cpu().numpy() - cos_o).max() < 1e-5


@gpu
def test_strip_width_and_block_size_do_not_change_bits():
    Q, G = 700, 2600
    N = Q + G
    s = make_retrieval_set(Q, G, 50, 4, dim=192, sigma=2.5, seed=33)
    qf, gf = unit(s.qf).cuda(), unit(s.gf).cuda()
    outs = []
    # 256- and 512-row strips, one strip per segment; the block budgets also give 128- to 700-row query blocks
    for rows in (256, 512, 4096):
        ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", block_bytes=strip_budget(N, 26, rows))
        cmc, mAP, info = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        outs.append((cmc, mAP, info["distmat"], ev._rr["rank"].clone(), ev._rr["S"].clone(), ev._rr["a_val"].clone()))
    for block_bytes in (128 * 12 * G, 384 * 12 * G):
        ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", block_bytes=block_bytes)
        cmc, mAP, info = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        outs.append((cmc, mAP, info["distmat"], ev._rr["rank"], ev._rr["S"], ev._rr["a_val"]))
    for cmc, mAP, d, rk, S, av in outs[1:]:
        assert np.array_equal(cmc, outs[0][0]) and mAP == outs[0][1]
        assert torch.equal(d, outs[0][2]) and torch.equal(rk, outs[0][3]) and torch.equal(S, outs[0][4])
        assert torch.equal(av, outs[0][5])


@gpu
def test_state_is_reused_for_the_same_queries():
    s = make_retrieval_set(200, 900, 20, 3, dim=128, sigma=2.5, seed=3)
    ev = RetrievalEvaluator(unit(s.gf).cuda(), s.g_pids, s.g_camids, rerank="gnn")
    assert (ev.k1, ev.k2) == (26, 7)
    qf = unit(s.qf).cuda()
    c1, m1, _ = ev.evaluate(qf, s.q_pids, s.q_camids)
    a_val = ev._rr["a_val"]
    c2, m2, _ = ev.evaluate(qf, s.q_pids, s.q_camids)
    assert ev._rr["a_val"] is a_val and np.array_equal(c1, c2) and m1 == m2
    ev.ranked_lists(qf, s.q_pids, s.q_camids)
    assert ev._rr["a_val"] is a_val
    qf.mul_(1.0)                              # a modified query tensor gets a new state
    ev.evaluate(qf, s.q_pids, s.q_camids)
    assert ev._rr["a_val"] is not a_val
    ev.k1, ev.k2 = 10, 3                      # so do other parameters
    c3, m3, i3 = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    fresh = RetrievalEvaluator(unit(s.gf).cuda(), s.g_pids, s.g_camids, rerank="gnn", k1=10, k2=3)
    c4, m4, i4 = fresh.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    assert np.array_equal(c3, c4) and m3 == m4 and torch.equal(i3["distmat"], i4["distmat"])


@gpu
def test_empty_query_set_as_with_k_reciprocal_reranking():
    s = make_retrieval_set(50, 300, 10, 3, dim=64, sigma=2.5, seed=4)

    def outcome(**kw):
        ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, **kw)
        try:
            cmc, mAP, _ = ev.evaluate(s.qf[:0].cuda(), s.q_pids[:0], s.q_camids[:0])
            return ("ok", cmc.tolist(), mAP)
        except Exception as e:                # noqa: BLE001 -- the k-reciprocal evaluator's own outcome is the reference
            return (type(e).__name__, str(e))
    gnn, krecip = outcome(rerank="gnn"), outcome(rerank=True)
    # both fail in the library on the zero-row block (at the first call that takes it): same exception, same code
    assert gnn[0] == krecip[0] and gnn[1].split(":")[0] == krecip[1].split(":")[0]
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank="gnn")
    idx, val = ev.ranked_lists(s.qf[:0].cuda(), k=5)
    assert idx.shape == (0, 5) and val.shape == (0, 5)


@gpu
def test_errors():
    s = make_retrieval_set(20, 60, 5, 2, dim=32, seed=1)
    gf = s.gf.cuda()
    with pytest.raises(ValueError, match="sharded"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", group=object())
    with pytest.raises(ValueError, match="from_host"):
        RetrievalEvaluator.from_host(s.gf, s.g_pids, s.g_camids, rerank="gnn")
    with pytest.raises(ValueError, match="precision"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, precision="fp32_simt", rerank="gnn")
    with pytest.raises(ValueError, match="integers"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", k1=2.5, k2=1)
    with pytest.raises(ValueError, match="integers"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", k1=20, k2=True)
    for k1, k2 in ((0, 1), (20, 0), (20, 21), (1025, 7)):
        with pytest.raises(ValueError, match="k2 <= k1"):
            RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", k1=k1, k2=k2)
    with pytest.raises(ValueError, match="rerank must be"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="knn")
    ev = RetrievalEvaluator(gf[:5], s.g_pids[:5], s.g_camids[:5], rerank="gnn", k1=20, k2=6)
    with pytest.raises(ValueError, match="exceeds"):
        ev.evaluate(s.qf[:3].cuda(), s.q_pids[:3], s.q_camids[:3])


@gpu
def test_beyond_both_dense_limits():
    """10 000 x 140 000 x 256: N = 150 000 > 65 535 rows of the dense propagation, and the dense A and B alone would
    take 8 N^2 ~ 180 GB (with the score matrix ~ 270 GB)."""
    Q, G, D, k1, k2 = 10000, 140000, 256, 26, 7
    N = Q + G
    s = make_retrieval_set(Q, G, 5000, 6, dim=D, sigma=2.75, seed=7)
    qf, gf = unit(s.qf).cuda(), unit(s.gf).cuda()
    block_bytes = 1 << 30
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", block_bytes=block_bytes)
    cmc, mAP, info = ev.evaluate(qf, s.q_pids, s.q_camids)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    rr = ev._rr
    state = sum(rr[k].numel() * rr[k].element_size() for k in ("rank", "S", "a_ptr", "a_col", "a_val", "g_ptr", "g_row", "g_val"))
    # the sparse state, the scratch (strips within block_bytes, then the index), the numeric phase's work buffer, the
    # distance block and its accumulators (within block_bytes) and the small rest: packed features, labels, rank stages
    assert peak <= state + rr["scratch_bytes"] + rr["work_bytes"] + block_bytes + (256 << 20), (peak, state)
    # neighbour lists of sampled rows against an independent contraction of those rows
    xu = torch.cat((qf, gf))
    rows = torch.cat((torch.arange(0, Q, 97), torch.arange(Q, N, 631), torch.tensor([N - 1]))).cuda()
    neg = _device_distmat(xu[rows], xu, "neg_dot")
    n = rows.numel()
    idx = torch.empty((n, k1), dtype=torch.int32, device="cuda")
    val = torch.empty((n, k1), dtype=torch.float32, device="cuda")
    _lib.call("ieee_topk", neg.data_ptr(), neg.stride(0), n, N, 0, None, None, None, None, k1, idx.data_ptr(), val.data_ptr(),
              _lib.stream())
    assert torch.equal(rr["rank"][rows], idx) and torch.equal(rr["S"][rows], val * val)
    # a few query rows of the output against an fp64 product from the exported CSR
    for q in (0, 4321, Q - 1):
        d = ev._gnn_block(q, q + 1)[0].double()
        aq = torch.zeros(N, dtype=torch.float64, device="cuda")
        p0, p1 = rr["a_ptr"][q].item(), rr["a_ptr"][q + 1].item()
        aq[rr["a_col"][p0:p1].long()] = rr["a_val"][p0:p1].double()
        g0 = rr["a_ptr"][Q].item()
        grow = torch.repeat_interleave(torch.arange(G, device="cuda"), rr["a_ptr"][Q:].diff())
        contrib = aq[rr["a_col"][g0:].long()] * rr["a_val"][g0:].double()
        ref = -torch.zeros(G, dtype=torch.float64, device="cuda").index_add_(0, grow, contrib)
        assert (d - ref).abs().max().item() <= 1e-6, q
    assert 0.0 < mAP <= 1.0


def test_scratch_size_query_limits():
    """The size query needs no GPU; out-of-range parameters give 0 and say why."""
    lib = _lib.load()
    assert lib.ieee_gnn_stream_scratch_bytes(100, 1000, 26, 1 << 30) > 0
    assert lib.ieee_gnn_stream_scratch_bytes(10, 10, 21, 1 << 30) == 0          # k1 > N
    assert b"exceeds" in lib.ieee_last_error()
    assert lib.ieee_gnn_stream_scratch_bytes(100, 1000, 1025, 1 << 30) == 0     # k1 > 1024
    assert b"k1 <= 1024" in lib.ieee_last_error()
    assert lib.ieee_gnn_stream_scratch_bytes(100, 1000, 0, 1 << 30) == 0
    assert lib.ieee_gnn_stream_scratch_bytes(1 << 19, (1 << 19) + 1, 26, 1 << 30) == 0   # N > 2^20
    assert b"exceeds" in lib.ieee_last_error()
    assert lib.ieee_gnn_stream_scratch_bytes(0, 1000, 26, 1 << 30) == 0
    assert b"bad shape" in lib.ieee_last_error()
    # the strips are a budget: one strip of 256 rows at least; beyond that the index (linear in N) may dominate
    small = lib.ieee_gnn_stream_scratch_bytes(1000, 9000, 26, 0)
    assert small >= 256 * 4 * (10016 + 26)
    assert lib.ieee_gnn_stream_scratch_bytes(1000, 9000, 26, 1 << 30) <= max(1 << 30, small) + (1 << 20)
