"""Streamed k-reciprocal re-ranking inside RetrievalEvaluator (rerank=True): the same bits as the dense path
(re_ranking_device on the three matrices the contraction writes for the same packed operands, then evaluate_device),
for every strip width, past the size the dense path can hold, and within the oracle's tolerance."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from ieee_b200 import _lib
from ieee_b200.engine import PackedFeatures, RetrievalEvaluator, packed_distmat
from ieee_b200.metrics.rank import evaluate_device, topk_ranked_list
from ieee_b200.testing import make_retrieval_set, market1501_shaped, rgbnt201_shaped
from ieee_b200.utils.rerank import re_ranking_device

gpu = pytest.mark.gpu


def strip_budget(Q, G, k1, width):
    """block_bytes that gives strips of `width` columns: the library sizes a strip column at
    4 * (Q + G and N rounded up to 32 + k1 + 1) bytes."""
    r32 = lambda x: (x + 31) // 32 * 32
    return width * 4 * (Q + r32(G) + r32(Q + G) + k1 + 1)


def dense_matrices(ev, qf, gf):
    """qg, qq, gg as the contraction writes them for the evaluator's packing (its centre, metric, precision)."""
    qpk = PackedFeatures(qf, ev.metric, ev.normalize, ev.precision, ev.center)
    gpk = PackedFeatures(gf, ev.metric, ev.normalize, ev.precision, ev.center)
    Q, G = qf.shape[0], gf.shape[0]
    dev = qf.device
    qg = packed_distmat(qpk, gpk, torch.empty((Q, G), dtype=torch.float32, device=dev))
    qq = packed_distmat(qpk, qpk, torch.empty((Q, Q), dtype=torch.float32, device=dev))
    gg = packed_distmat(gpk, gpk, torch.empty((G, G), dtype=torch.float32, device=dev))
    return qg, qq, gg


def check_identical(s, k1=20, k2=6, lam=0.3, metric="euclidean", normalize=False, dtype=torch.float32, block_bytes=None,
                    max_rank=20):
    qf, gf = s.qf.cuda().to(dtype), s.gf.cuda().to(dtype)
    kw = {} if block_bytes is None else {"block_bytes": block_bytes}
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, metric, normalize, max_rank=max_rank, rerank=True, k1=k1, k2=k2,
                            lambda_value=lam, **kw)
    cmc, mAP, info = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    dense = re_ranking_device(*dense_matrices(ev, qf, gf), k1=k1, k2=k2, lambda_value=lam)
    cmc_d, summary, st = evaluate_device(dense, s.q_pids, s.g_pids, s.q_camids, s.g_camids, max_rank)
    assert torch.equal(info["distmat"], dense)
    assert np.array_equal(cmc, cmc_d.cpu().numpy())
    assert mAP == float(summary.mAP) and info["mINP"] == float(summary.mINP)
    assert torch.equal(info["ap"], st.ap) and torch.equal(info["first"], st.first)
    return ev, qf, info, dense


@gpu
def test_rgbnt201_shape_self_duplicates():
    """Config C3 (query set == gallery set: every query has an exact duplicate in the gallery)."""
    check_identical(rgbnt201_shaped())


@gpu
@pytest.mark.parametrize("Q,G,k1,k2", [(5, 16, 20, 6), (8, 13, 19, 20), (1, 30, 29, 3), (30, 1, 20, 21)])
def test_tiny_shapes_k1_near_n(Q, G, k1, k2):
    s = make_retrieval_set(Q, G, 4, 2, dim=48, sigma=1.5, seed=Q * 100 + G)
    # two identities, queries and gallery on different cameras: every query keeps all G items (no junk) and
    # identity 0 always has a match
    s.q_pids, s.g_pids = np.arange(Q, dtype=np.int64) % 2, np.arange(G, dtype=np.int64) % 2
    s.q_camids, s.g_camids = np.zeros(Q, dtype=np.int64), np.ones(G, dtype=np.int64)
    check_identical(s, k1=k1, k2=k2, max_rank=min(5, G))


@gpu
def test_many_strips_ragged_query_count():
    """1000 x 5003: 256-column strips (Q is not a multiple of 256) and 512-row query blocks."""
    s = make_retrieval_set(1000, 5003, 60, 4, dim=320, sigma=2.5, seed=13, distractor_frac=0.1)
    check_identical(s, block_bytes=strip_budget(1000, 5003, 20, 256))


@gpu
@pytest.mark.parametrize("k1,k2,lam", [(20, 1, 0.3), (30, 8, 0.3), (12, 4, 0.0), (6, 3, 1.0)])
def test_parameters(k1, k2, lam):
    s = make_retrieval_set(420, 1900, 40, 4, dim=256, sigma=2.5, seed=k1 + k2)
    check_identical(s, k1=k1, k2=k2, lam=lam)


@gpu
def test_cosine_normalized():
    s = make_retrieval_set(300, 1700, 30, 4, dim=384, sigma=2.5, seed=21)
    check_identical(s, metric="cosine", normalize=True)


@gpu
def test_bf16():
    s = make_retrieval_set(300, 1700, 30, 4, dim=384, sigma=2.5, seed=22)
    ev, _, _, _ = check_identical(s, dtype=torch.bfloat16)
    assert ev.precision == "bf16"


@gpu
def test_market_shaped():
    s = market1501_shaped()
    ev, qf, info, dense = check_identical(s)
    # ranked_lists on a re-ranking evaluator lists what was evaluated
    idx, val = ev.ranked_lists(qf, s.q_pids, s.q_camids, k=10)
    idx_d, val_d = topk_ranked_list(dense, s.q_pids, s.g_pids, s.q_camids, s.g_camids, k=10)
    assert torch.equal(idx.cpu(), torch.as_tensor(idx_d).cpu()) and torch.equal(val.cpu(), torch.as_tensor(val_d).cpu())


@gpu
def test_strip_width_does_not_change_bits():
    Q, G = 700, 2600
    s = make_retrieval_set(Q, G, 50, 4, dim=192, sigma=2.5, seed=33)
    outs = []
    for width in (256, 512, 4096):          # 4096: one strip over the queries and one over the gallery
        ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True, block_bytes=strip_budget(Q, G, 20, width))
        cmc, mAP, info = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True)
        outs.append((cmc, mAP, info["distmat"], ev._rr["colmax"].clone(), ev._rr["rank"].clone()))
    for cmc, mAP, d, cm, rk in outs[1:]:
        assert np.array_equal(cmc, outs[0][0]) and mAP == outs[0][1]
        assert torch.equal(d, outs[0][2]) and torch.equal(cm, outs[0][3]) and torch.equal(rk, outs[0][4])


@gpu
def test_state_is_reused_for_the_same_queries():
    s = make_retrieval_set(200, 900, 20, 3, dim=128, sigma=2.5, seed=3)
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True)
    qf = s.qf.cuda()
    c1, m1, _ = ev.evaluate(qf, s.q_pids, s.q_camids)
    ws = ev._rr["ws"]
    c2, m2, _ = ev.evaluate(qf, s.q_pids, s.q_camids)
    assert ev._rr["ws"] is ws and np.array_equal(c1, c2) and m1 == m2
    qf.mul_(1.0)                              # a modified query tensor gets a new state
    ev.evaluate(qf, s.q_pids, s.q_camids)
    assert ev._rr["ws"] is not ws
    ev.k1, ev.k2 = 10, 3                      # so do other parameters
    c3, m3, i3 = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    fresh = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True, k1=10, k2=3)
    c4, m4, i4 = fresh.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    assert np.array_equal(c3, c4) and m3 == m4 and torch.equal(i3["distmat"], i4["distmat"])


@gpu
def test_empty_query_set_as_without_reranking():
    s = make_retrieval_set(50, 300, 10, 3, dim=64, sigma=2.5, seed=4)

    def outcome(**kw):
        ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, **kw)
        try:
            cmc, mAP, _ = ev.evaluate(s.qf[:0].cuda(), s.q_pids[:0], s.q_camids[:0])
            return ("ok", cmc.tolist(), mAP)
        except Exception as e:                # noqa: BLE001 -- the plain evaluator's own outcome is the reference
            return (type(e).__name__, str(e))
    assert outcome(rerank=True) == outcome()


@gpu
def test_beyond_the_dense_limit():
    """Q = 4096, G = 196 608: the dense path would need 8 N^2 ~ 320 GB."""
    Q, G, D, k1 = 4096, 196608, 64, 20
    s = make_retrieval_set(Q, G, 2000, 6, dim=D, sigma=1.2, seed=7)
    qf, gf = s.qf.cuda(), s.gf.cuda()
    block_bytes = 1 << 30
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank=True, block_bytes=block_bytes)
    cmc, mAP, _ = ev.evaluate(qf, s.q_pids, s.q_camids)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    ws = _lib.load().ieee_rerank_stream_workspace_bytes(Q, G, k1, 6)
    # the workspace, the block budget (first the strips, then the distance block and the blend's accumulators) and
    # the small rest: packed features, colmax and rank, labels, rank stages
    assert peak <= ws + block_bytes + (256 << 20), (peak, ws)
    # colmax and the first k1 + 1 neighbours of sampled samples, recomputed from 256-aligned contraction slices
    colmax, rank = ev._rr["colmax"], ev._rr["rank"]
    qpk = PackedFeatures(qf, "euclidean", False, ev.precision, ev.center)
    gpk = PackedFeatures(gf, "euclidean", False, ev.precision, ev.center)
    for i in (0, 255, 1000, Q - 1, Q, Q + 70001, Q + G - 1):
        gal = i >= Q
        c = i - Q if gal else i
        c0 = c // 256 * 256
        feats = gf if gal else qf
        spk = PackedFeatures(feats[c0: c0 + 256], "euclidean", False, ev.precision, ev.center)
        n = spk.rows
        top = packed_distmat(qpk, spk, torch.empty((Q, n), device="cuda"))[:, c - c0]
        if gal:
            bot = packed_distmat(gpk, spk, torch.empty((G, n), device="cuda"))[:, c - c0]
        else:
            bot = packed_distmat(spk, gpk, torch.empty((n, G), device="cuda"))[c - c0]
        raw = torch.cat([top, bot])
        sq = raw * raw
        cm = sq.max()
        assert colmax[i].item() == cm.item(), i
        order = torch.sort(sq / cm, stable=True).indices[: k1 + 1]
        assert torch.equal(rank[i].long(), order), i
    plain = RetrievalEvaluator(gf, s.g_pids, s.g_camids)
    _, mAP_plain, _ = plain.evaluate(qf, s.q_pids, s.q_camids)
    assert mAP > mAP_plain, (mAP, mAP_plain)


@gpu
def test_cpu_restatement():
    """Within 1e-5 of the oracle's re_ranking on the same three distance matrices."""
    s = make_retrieval_set(60, 340, 12, 3, dim=96, sigma=2.0, seed=9)
    qf, gf = s.qf.cuda(), s.gf.cuda()
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank=True, k1=10, k2=4, lambda_value=0.2)
    _, _, info = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    qg, qq, gg = (m.cpu().numpy() for m in dense_matrices(ev, qf, gf))
    out_o = R.re_ranking(qg, qq, gg, k1=10, k2=4, lambda_value=0.2)
    assert np.abs(info["distmat"].cpu().numpy() - out_o).max() <= 1e-5


@gpu
def test_errors():
    s = make_retrieval_set(20, 60, 5, 2, dim=32, seed=1)
    gf = s.gf.cuda()
    with pytest.raises(ValueError, match="sharded"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank=True, group=object())
    with pytest.raises(ValueError, match="from_host"):
        RetrievalEvaluator.from_host(s.gf, s.g_pids, s.g_camids, rerank=True)
    for k1, k2 in ((0, 1), (511, 6), (20, 0), (20, 22), (100, 10), (2.5, 1), (20, True)):
        with pytest.raises(ValueError, match="k1|k2|sort"):
            RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank=True, k1=k1, k2=k2)
    with pytest.raises(ValueError, match="precision"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, precision="fp32_simt", rerank=True)
    ev = RetrievalEvaluator(gf[:5], s.g_pids[:5], s.g_camids[:5], rerank=True, k1=20, k2=6)
    with pytest.raises(ValueError, match="exceeds"):
        ev.evaluate(s.qf[:3].cuda(), s.q_pids[:3], s.q_camids[:3])


def test_workspace_size_is_linear_in_n():
    """The size query needs no GPU; at a fixed strip width it grows linearly in N = Q + G."""
    lib = _lib.load()
    size = lambda n: lib.ieee_rerank_stream_workspace_bytes(n // 8, n - n // 8, 20, 6)
    s1, s2, s4, s8 = size(1 << 16), size(1 << 17), size(1 << 18), size(1 << 19)
    assert s1 > 0
    per_n = (s8 - s4) / (1 << 18)
    assert abs((s2 - s1) / (1 << 16) - per_n) <= 1e-3 * per_n and abs((s4 - s2) / (1 << 17) - per_n) <= 1e-3 * per_n
    assert lib.ieee_rerank_stream_workspace_bytes(100, 1000, 20, 22) == 0     # k2 > k1 + 1
    assert lib.ieee_rerank_stream_workspace_bytes(1 << 23, 1 << 23, 20, 6) == 0   # N = 2^24
    assert lib.ieee_rerank_stream_workspace_bytes(5, 10, 20, 6) == 0          # k1 + 1 > N
    assert b"exceeds" in lib.ieee_last_error()
    # the strips' scratch is a budget, not a function of N: at least one 256-column strip, at most the budget
    assert lib.ieee_rerank_stream_scratch_bytes(1 << 12, 1 << 18, 20, 1 << 30) <= (1 << 30) + (8 << 20)
    assert lib.ieee_rerank_stream_scratch_bytes(5, 10, 20, 1 << 30) == 0
