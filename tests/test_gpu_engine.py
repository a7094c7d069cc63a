"""GPU parity: the device-resident evaluation path (engine.py:391-425) incl. blocking and the padded scratch pitch."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from ieee_b200.engine import RetrievalEvaluator, evaluate
from ieee_b200.testing import make_retrieval_set, rgbnt201_shaped

pytestmark = pytest.mark.gpu


def oracle_eval(s, metric="euclidean", normalize=False, max_rank=20, distmat=None):
    qf, gf = s.qf, s.gf
    if normalize:
        qf, gf = torch.nn.functional.normalize(qf, p=2, dim=1), torch.nn.functional.normalize(gf, p=2, dim=1)
    d = R.compute_distance_matrix(qf, gf, metric).numpy() if distmat is None else distmat
    return R.evaluate_rank(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, max_rank=max_rank)


@pytest.mark.parametrize("metric,normalize", [("euclidean", False), ("cosine", False), ("euclidean", True)])
def test_evaluate_matches_oracle_on_own_distmat(metric, normalize):
    """Rank order is only well posed on identical distance bits: feed the oracle the GPU's own distmat."""
    s = make_retrieval_set(300, 2001, 40, 4, dim=512, sigma=2.5, seed=31, distractor_frac=0.1)
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, metric, normalize)
    cmc, mAP, info = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True)
    d = info["distmat"].cpu().numpy()
    cmc_o, map_o = oracle_eval(s, distmat=d)
    assert np.array_equal(cmc, cmc_o) and abs(mAP - map_o) < 1e-9
    # and the metrics agree with the pure-CPU pipeline up to distance rounding
    cmc_c, map_c = oracle_eval(s, metric, normalize)
    assert abs(mAP - map_c) < 2e-3 and np.abs(cmc - cmc_c).max() < 1e-2


def test_query_blocking_is_invisible():
    s = make_retrieval_set(700, 900, 25, 3, dim=128, sigma=2.0, seed=8)
    one = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids)
    many = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, block_bytes=128 * 900 * 4)   # 128-query blocks
    c1, m1, i1 = one.evaluate(s.qf.cuda(), s.q_pids, s.q_camids)
    c2, m2, i2 = many.evaluate(s.qf.cuda(), s.q_pids, s.q_camids)
    assert np.array_equal(c1, c2) and m1 == m2
    assert torch.equal(i1["first"], i2["first"]) and torch.equal(i1["ap"], i2["ap"])


def test_engine_prints_reference_lines(capsys):
    s = rgbnt201_shaped()
    cmc, mAP = evaluate(s.qf, s.gf, s.q_pids, s.g_pids, s.q_camids, s.g_camids, ranks=[1, 5, 10], dataset_name="RGBNT201")
    out = capsys.readouterr().out
    assert "Computing distance matrix with metric=euclidean ..." in out and "** Results **" in out
    assert "mAP: {:.2%}".format(mAP) in out and "Rank-1  : {:.2%}".format(cmc[0]) in out
    with pytest.raises(ValueError):
        evaluate(s.qf, s.gf, s.q_pids, s.g_pids, s.q_camids, s.g_camids, dist_metric="manhattan")


def test_streamed_host_gallery_equals_resident():
    """RetrievalEvaluator.from_host (chunked PCIe copy overlapped with the contraction) == device-resident path."""
    s = make_retrieval_set(260, 1500, 30, 4, dim=256, sigma=2.5, seed=44)
    res = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids)
    c1, m1, i1 = res.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True)
    host = RetrievalEvaluator.from_host(s.gf.pin_memory(), s.g_pids, s.g_camids, num_chunks=3)
    c2, m2, i2 = host.evaluate(s.qf.pin_memory(), s.q_pids, s.q_camids, return_distmat=True)
    assert torch.equal(i1["distmat"], i2["distmat"]) and np.array_equal(c1, c2) and m1 == m2
    c3, m3 = evaluate(s.qf, s.gf, s.q_pids, s.g_pids, s.q_camids, s.g_camids, verbose=False)      # pageable host tensors
    assert np.array_equal(c1, c3) and m1 == m3


@pytest.mark.parametrize("one_call", [True, False])
def test_capacity_memo_is_checked_not_trusted(one_call):
    """The list-capacity memo is keyed by label tensor identity + version; a stale (too small) hint is caught by the
    gather kernel's overflow flag and the evaluation is redone with the exact capacity."""
    from ieee_b200 import engine
    s = make_retrieval_set(200, 1500, 20, 3, dim=128, sigma=2.0, seed=9)
    dev = torch.device("cuda")
    lab = [torch.from_numpy(x).to(dev) for x in (s.q_pids, s.q_camids, s.g_pids, s.g_camids)]
    ev = RetrievalEvaluator(s.gf.cuda(), lab[2], lab[3])
    c1, m1, i1 = ev.evaluate(s.qf.cuda(), lab[0], lab[1], one_call=one_call)
    key = [k for k in engine._CAP_MEMO if k[0] == ev._label_keys][0]
    assert engine._CAP_MEMO[key][0] == i1["cap"]
    c2, m2, i2 = ev.evaluate(s.qf.cuda(), lab[0], lab[1], one_call=one_call)              # memo hit: same result, no capacity query
    assert np.array_equal(c1, c2) and m1 == m2
    engine._CAP_MEMO[key] = (2, 0)                                       # poison the hint: far too small
    c3, m3, i3 = ev.evaluate(s.qf.cuda(), lab[0], lab[1], one_call=one_call)
    assert np.array_equal(c1, c3) and m1 == m3 and i3["cap"] == i1["cap"]
    if not one_call:
        # the staged path also remembers the longest merged list (row width of the count table); too narrow a
        # hint is reported by the count kernel and the evaluation is redone
        ev.evaluate(s.qf.cuda(), lab[0], lab[1], one_call=False)
        cap, width = engine._CAP_MEMO[key]
        assert 1 <= width <= cap
        engine._CAP_MEMO[key] = (cap, 1)
        c4, m4, _ = ev.evaluate(s.qf.cuda(), lab[0], lab[1], one_call=False)
        assert np.array_equal(c1, c4) and m1 == m4
    lab[0][0] += 0                                                       # in-place op bumps the version: key changes
    assert engine._tensor_key(lab[0]) != key[1]


def test_one_call_path_equals_staged_path():
    """ieee_retrieve_eval_prepared (one foreign call per evaluation) == the staged path kernel by kernel; mINP vs the
    oracle's sort form on the GPU's own distance bits."""
    s = make_retrieval_set(333, 2500, 45, 5, dim=320, sigma=2.5, seed=77, distractor_frac=0.15)
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids)
    c1, m1, i1 = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True, one_call=True)
    c2, m2, i2 = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True, one_call=False)
    assert torch.equal(i1["distmat"], i2["distmat"])
    assert np.array_equal(c1, c2) and m1 == m2 and i1["mINP"] == i2["mINP"] and i1["num_ties"] == i2["num_ties"]
    assert torch.equal(i1["first"], i2["first"]) and torch.equal(i1["ap"], i2["ap"])
    d = i1["distmat"].cpu().numpy()
    cmc_o, map_o = oracle_eval(s, distmat=d)
    assert np.array_equal(c1, cmc_o) and abs(m1 - map_o) < 1e-9
    minp_o = R.mean_inverse_negative_penalty(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    assert abs(i1["mINP"] - minp_o) < 1e-12


def test_one_call_path_checks_the_capacity_hint():
    from ieee_b200 import engine
    s = make_retrieval_set(150, 1200, 15, 3, dim=128, sigma=2.0, seed=10)
    dev = torch.device("cuda")
    lab = [torch.from_numpy(x).to(dev) for x in (s.q_pids, s.q_camids, s.g_pids, s.g_camids)]
    ev = RetrievalEvaluator(s.gf.cuda(), lab[2], lab[3])
    c1, m1, i1 = ev.evaluate(s.qf.cuda(), lab[0], lab[1])
    key = [k for k in engine._CAP_MEMO if k[0] == ev._label_keys][0]
    engine._CAP_MEMO[key] = (3, 0)                                       # stale, too small
    c2, m2, i2 = ev.evaluate(s.qf.cuda(), lab[0], lab[1])
    assert np.array_equal(c1, c2) and m1 == m2 and i2["cap"] == i1["cap"] and engine._CAP_MEMO[key][0] == i1["cap"]


@pytest.mark.parametrize("metric,normalize", [("euclidean", False), ("cosine", False), ("euclidean", True)])
def test_one_call_equals_staged_path_per_metric(metric, normalize):
    """The one-call path against the staged path for every metric, with ~16 gallery items per identity and queries
    whose identity the gallery does not have: bit-identical CMC, mAP, per-query AP / first hit, mINP and tie count."""
    s = make_retrieval_set(333, 2500, 160, 5, dim=320, sigma=2.5, seed=77)      # ~16 gallery items per identity
    s.q_pids[:3] = 10 ** 6                                               # identities the gallery does not have
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, metric, normalize)
    c1, m1, i1 = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, one_call=True)
    c2, m2, i2 = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, one_call=False)
    assert np.array_equal(c1, c2) and m1 == m2 and i1["mINP"] == i2["mINP"] and i1["num_ties"] == i2["num_ties"]
    assert torch.equal(i1["first"], i2["first"]) and torch.equal(i1["ap"], i2["ap"]) and i1["num_valid"] == i2["num_valid"] == 330


def test_one_call_equals_staged_path_full_size_with_duplicates():
    """Market-shaped, feature width 2304, gallery rows duplicated (bit-equal distances: ties by gallery index) and the
    query set containing gallery rows (exact zeros: the near-duplicate fix-up): the one-call path against the staged
    path, and both against the oracle on the GPU's own distances."""
    from ieee_b200.testing import market1501_shaped
    s = market1501_shaped(seed=3, num_q=700)
    gf, g_pids, g_camids = s.gf.clone(), s.g_pids.copy(), s.g_camids.copy()
    small = np.isin(s.g_pids, np.nonzero(np.bincount(s.g_pids) <= 16)[0])  # identities of at most 16 items
    src = np.nonzero(small[:8000])[0][:1000]
    dst = 15912 - np.arange(src.size)
    dst = dst[~np.isin(dst, src)]
    src = src[: dst.size]
    gf[dst] = gf[src]
    g_pids[dst], g_camids[dst] = g_pids[src], (g_camids[src] + 1) % 6
    qf = s.qf.clone()
    twins = np.nonzero(g_pids != 0)[0][100:150]                          # (pid 0 = distractors: 2 680 of them, no query)
    qf[:50] = gf[twins]                                                   # queries identical to gallery rows
    q_pids, q_camids = s.q_pids.copy(), s.q_camids.copy()
    q_pids[:50], q_camids[:50] = g_pids[twins], (g_camids[twins] + 2) % 6
    ev = RetrievalEvaluator(gf.cuda(), g_pids, g_camids)
    c1, m1, i1 = ev.evaluate(qf.cuda(), q_pids, q_camids, return_distmat=True, one_call=True)
    c2, m2, i2 = ev.evaluate(qf.cuda(), q_pids, q_camids, return_distmat=True, one_call=False)
    assert torch.equal(i1["distmat"], i2["distmat"])
    assert i2["num_ties"] > 0 and i1["num_ties"] == i2["num_ties"]
    assert np.array_equal(c1, c2) and m1 == m2 and torch.equal(i1["first"], i2["first"]) and torch.equal(i1["ap"], i2["ap"])
    d = i1["distmat"].cpu().numpy()
    assert (d[np.arange(50), twins] == 0).all()                          # the duplicates really are at distance 0
    cmc_o, map_o = R.evaluate_rank(d, q_pids, g_pids, q_camids, g_camids, max_rank=20)
    assert np.array_equal(c1, cmc_o) and abs(m1 - map_o) < 1e-9
