"""GPU parity: evaluate_rank / top-k through the drop-in API and the C ABI vs the CPU oracle."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import ref, restatement as R
from ieee_b200 import _lib
from ieee_b200.metrics import evaluate_rank
from ieee_b200.metrics.rank import evaluate_device, topk_ranked_list
from ieee_b200.testing import make_retrieval_set, market1501_shaped, rgbnt201_shaped

pytestmark = pytest.mark.gpu


def check_against_oracle(d, qp, gp, qc, gc, max_rank=20):
    cmc_o, map_o = R.evaluate_rank(d, qp, gp, qc, gc, max_rank=max_rank)          # stable ties (gallery index)
    cmc, mAP = evaluate_rank(d, qp, gp, qc, gc, max_rank=max_rank)
    assert isinstance(cmc, np.ndarray) and cmc.dtype == np.float32 and isinstance(mAP, float)
    assert np.array_equal(cmc, cmc_o), "CMC must be bit-exact"
    assert abs(mAP - map_o) < 1e-9, (mAP, map_o)                                   # bar: 1e-6
    return cmc, mAP


@pytest.mark.parametrize("name", ["rank_cython_shape.npz", "rank_clustered.npz", "rank_ties_stable.npz"])
def test_golden_rank(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    cmc, mAP = evaluate_rank(g["distmat"], g["q_pids"], g["g_pids"], g["q_camids"], g["g_camids"],
                             max_rank=int(g["max_rank"]))
    assert np.array_equal(cmc, g["cmc"]) and abs(mAP - float(g["mAP"])) < 1e-9


def test_tie_count_reported(golden_dir):
    g = np.load(os.path.join(golden_dir, "rank_ties_stable.npz"))
    d = torch.from_numpy(g["distmat"]).cuda()
    _, summary, st = evaluate_device(d, g["q_pids"], g["g_pids"], g["q_camids"], g["g_camids"], 20)
    # oracle tie count: (relevant r, kept non-relevant g) pairs with equal distance
    want = 0
    for q in range(d.shape[0]):
        same = g["g_pids"] == g["q_pids"][q]
        junk = same & (g["g_camids"] == g["q_camids"][q])
        rel = same & ~junk
        other = ~same
        want += int((g["distmat"][q][rel][:, None] == g["distmat"][q][other][None, :]).sum())
    assert summary.num_ties == want and want > 0
    g2 = np.load(os.path.join(golden_dir, "rank_clustered.npz"))
    _, s2, _ = evaluate_device(torch.from_numpy(g2["distmat"]).cuda(), g2["q_pids"], g2["g_pids"], g2["q_camids"],
                               g2["g_camids"], 20)
    assert s2.num_ties == 0


def test_rgbnt201_shaped_with_natural_ties():
    s = rgbnt201_shaped()
    d = R.compute_distance_matrix(s.qf, s.gf).numpy()          # identical distmat bits for both sides
    check_against_oracle(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    if ref.available() and R.count_row_ties(d) == 0:
        cmc_r, map_r = ref.evaluate_rank(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
        cmc, mAP = evaluate_rank(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
        assert np.array_equal(cmc, cmc_r) and abs(mAP - map_r) < 1e-9


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_clustered_sets_per_query_positions(metric):
    s = make_retrieval_set(200, 3000, 40, 4, dim=256, sigma=2.5, seed=12, distractor_frac=0.15)
    s.q_pids[:5] = 10 ** 12 + 7                                # int64 ids beyond int32, absent from the gallery
    d = R.compute_distance_matrix(s.qf, s.gf, metric).numpy()
    check_against_oracle(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, max_rank=50)
    # per-query intermediates: first-hit rank and AP
    _, _, info = R.eval_market1501(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, 50, return_info=True)
    _, summary, st = evaluate_device(torch.from_numpy(d).cuda(), s.q_pids, s.g_pids, s.q_camids, s.g_camids, 50)
    first = st.first.cpu().numpy()
    assert np.array_equal(first, info["first_hit"])
    ap = st.ap.cpu().numpy()[first >= 0]
    np.testing.assert_allclose(ap, info["ap"], rtol=0, atol=1e-12)
    assert summary.num_valid == info["num_valid"] == 195


def test_heavy_ties_and_special_values():
    rng = np.random.RandomState(3)
    d = rng.randint(0, 12, size=(64, 500)).astype(np.float32)      # ~40 equal values per level
    d[3, :50] = np.inf
    d[4, 10:30] = -np.inf
    d[5, ::7] = np.nan                                             # NaN ranks last (NumPy order)
    d[6, :] = 1.0                                                  # every distance equal: pure index order
    d[7, ::2] = -0.0
    d[7, 1::2] = 0.0                                               # -0.0 == +0.0
    qp, gp = rng.randint(0, 10, 64), rng.randint(0, 10, 500)
    qc, gc = rng.randint(0, 3, 64), rng.randint(0, 3, 500)
    check_against_oracle(d, qp, gp, qc, gc, max_rank=20)


_team_ties = []


@pytest.mark.parametrize("team", [1, 2, 4, 8])
def test_count_team_sizes_give_identical_results(team):
    """Rows of 4 K .. 64 K columns are streamed by 1, 2, 4 or 8 warps per query (ieee_set_count_team): ragged row
    length, heavy ties, NaN / inf, invalid queries, a query count that does not fill the last CTA."""
    lib = _lib.load()
    rng = np.random.RandomState(77)
    Q, G = 157, 9001
    d = np.round(rng.rand(Q, G) * 300).astype(np.float32)          # ~30 equal values per level
    d[3, ::11] = np.nan
    d[4, :40] = np.inf
    d[5, 100:140] = -np.inf
    d[6, :] = 2.0
    qp, gp = rng.randint(0, 60, Q), rng.randint(0, 64, G)          # identities 60 .. 63 are never queried
    qp[7] = 10 ** 12                                               # not in the gallery: invalid query
    qc, gc = rng.randint(0, 3, Q), rng.randint(0, 3, G)
    prev = lib.ieee_set_count_team(team)
    try:
        assert lib.ieee_set_count_team(-1) == team
        check_against_oracle(d, qp, gp, qc, gc, max_rank=20)
        dd = torch.from_numpy(d).cuda()
        _, summary, st = evaluate_device(dd, qp, gp, qc, gc, 20)
        _, _, info = R.eval_market1501(d, qp, gp, qc, gc, 20, return_info=True)
        assert np.array_equal(st.first.cpu().numpy(), info["first_hit"])
        _team_ties.append(int(summary.num_ties))
        assert len(set(_team_ties)) == 1 and _team_ties[0] > 0              # the tie statistic does not depend on the team size either
    finally:
        lib.ieee_set_count_team(prev)


@pytest.mark.parametrize("G", [700, 70000])        # warp-per-query kernel / CTA-per-query kernel
def test_degenerate_threshold_spans(G):
    """One relevant item per query, two at the same distance, two one ulp apart, a huge span: the cell table must
    stay exact when (d_max - d_min) of the relevant items is 0, tiny or enormous."""
    rng = np.random.RandomState(G)
    Q = 24
    d = (rng.rand(Q, G) * 50 + 100).astype(np.float32)
    gp = rng.randint(1000, 2000, G)                    # nobody's identity ...
    gc = rng.randint(0, 3, G)
    qp, qc = np.arange(Q), np.zeros(Q, int)
    for q in range(Q):
        cols = rng.choice(G, 3, replace=False)
        kind = q % 6
        if kind == 0:                                   # exactly one relevant item
            gp[cols[0]] = q; gc[cols[0]] = 1
        elif kind == 1:                                 # two relevant items, equal distance (span 0, R = 2)
            gp[cols[:2]] = q; gc[cols[:2]] = 1
            d[q, cols[1]] = d[q, cols[0]]
        elif kind == 2:                                 # two relevant items one ulp apart
            gp[cols[:2]] = q; gc[cols[:2]] = 1
            d[q, cols[1]] = np.nextafter(d[q, cols[0]], np.float32(1e9))
        elif kind == 3:                                 # enormous span: one relevant item at 1e30
            gp[cols[:2]] = q; gc[cols[:2]] = 1
            d[q, cols[1]] = 1e30
        elif kind == 4:                                 # one relevant item tied with many others
            gp[cols[0]] = q; gc[cols[0]] = 1
            d[q, ::5] = d[q, cols[0]]
        else:                                           # one relevant + one junk item
            gp[cols[:2]] = q; gc[cols[0]] = 1; gc[cols[1]] = 0
    check_against_oracle(d, qp, gp, qc, gc, max_rank=20)


@pytest.mark.parametrize("G", [3000, 70001])
def test_long_relevant_lists(G):
    """Hundreds of relevant items per query (more than the 128 the private-counter kernels hold): the CTA-per-query
    kernel with shared atomics, incl. ties and rows longer than 64K."""
    rng = np.random.RandomState(G)
    Q = 20
    d = rng.rand(Q, G).astype(np.float32)
    d[:, ::9] = np.round(d[:, ::9] * 8) / 8                      # ties between relevant and other items
    n_pid = 6 if G < 10000 else 14               # ~500 / ~5000 gallery items per identity (the kernel holds 8192)
    gp, gc = rng.randint(0, n_pid, G), rng.randint(0, 3, G)
    qp, qc = rng.randint(0, n_pid, Q), rng.randint(0, 3, Q)
    check_against_oracle(d, qp, gp, qc, gc, max_rank=20)
    if G > 10000:                                # beyond the shared-memory budget: a clear error, never a wrong answer
        with pytest.raises(_lib.IeeeB200Error, match="shared-memory budget"):
            evaluate_rank(d, qp % 4, gp % 4, qc, gc, max_rank=20)


def test_unaligned_rows_and_device_input():
    s = make_retrieval_set(33, 1001, 12, 3, dim=64, sigma=2.0, seed=6)     # G odd: rows start at any 4-byte offset
    d = R.compute_distance_matrix(s.qf, s.gf).numpy()
    cmc_o, map_o = R.evaluate_rank(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    padded = torch.zeros(33, 1003).cuda()
    padded[:, 1:1002] = torch.from_numpy(d).cuda()
    cmc, mAP = evaluate_rank(padded[:, 1:1002], torch.from_numpy(s.q_pids).cuda(), s.g_pids.astype(np.int32),
                             s.q_camids.tolist(), torch.from_numpy(s.g_camids))
    assert np.array_equal(cmc, cmc_o) and abs(mAP - map_o) < 1e-9


def test_max_rank_clamp_and_errors(capsys):
    rng = np.random.RandomState(0)
    d = rng.rand(6, 12).astype(np.float32)
    qp, gp = np.arange(6) % 3, np.arange(12) % 3
    qc, gc = np.zeros(6, int), np.ones(12, int)
    cmc, mAP = evaluate_rank(d, qp, gp, qc, gc, max_rank=50)               # rank.py:110-115
    assert cmc.shape == (12,) and "quite small" in capsys.readouterr().out
    assert np.array_equal(cmc, R.evaluate_rank(d, qp, gp, qc, gc, max_rank=50)[0])
    with pytest.raises(AssertionError, match="all query identities do not appear in gallery"):   # rank.py:165
        evaluate_rank(d, qp + 100, gp, qc, gc)
    for empty in (np.zeros((0, 12), np.float32), np.zeros((6, 0), np.float32)):                 # empty query / gallery set
        with pytest.raises(AssertionError, match="all query identities do not appear in gallery"):
            evaluate_rank(empty, qp[:empty.shape[0]], gp[:empty.shape[1]], qc[:empty.shape[0]], gc[:empty.shape[1]])
    with pytest.raises(TypeError):                                                              # rank.py:236-239
        evaluate_rank(d, qp, gp, qc, gc, use_metric_cuhk03=True)
    # kept lists shorter than max_rank (rank.py:150,167).  All but 2 gallery items are junk for camera-0 queries:
    gc2 = np.zeros(12, int); gp2 = np.zeros(12, int); gc2[:2] = 1
    # (a) EVERY valid query keeps the same 2 items: the reference stacks rows of length 2 and returns 2 ranks.  Both
    # kept items are relevant, so its result is CMC [1, 1] and mAP 1 whatever the order (the compiled reference's
    # answer, kept here so that the check runs without it; still compared live where oracle/_ref is built)
    cmc_u, map_u = evaluate_rank(d, np.zeros(6, int), gp2, np.zeros(6, int), gc2, max_rank=5)
    ref_cmc, ref_map = np.ones(2, np.float32), 1.0
    assert cmc_u.shape == (2,) and np.array_equal(cmc_u, ref_cmc) and abs(map_u - ref_map) < 1e-9
    cmc_r, map_r = R.evaluate_rank(d, np.zeros(6, int), gp2, np.zeros(6, int), gc2, max_rank=5, stable=False)
    assert np.array_equal(cmc_r, ref_cmc) and abs(map_r - ref_map) < 1e-9
    # (b) lists of different length (camera-1 queries keep 10): the reference dies building a ragged array (ValueError,
    # rank.py:167, which the restatement repeats line for line)
    qc2 = np.array([0, 1, 0, 1, 0, 1])
    with pytest.raises(ValueError):
        R.evaluate_rank(d, np.zeros(6, int), gp2, qc2, gc2, max_rank=5, stable=False)
    if ref.available():
        cmc_r, map_r = ref.evaluate_rank(d, np.zeros(6, int), gp2, np.zeros(6, int), gc2, max_rank=5, use_cython=False)
        assert np.array_equal(cmc_r, ref_cmc) and abs(map_r - ref_map) < 1e-9
        with pytest.raises(ValueError):
            ref.evaluate_rank(d, np.zeros(6, int), gp2, qc2, gc2, max_rank=5, use_cython=False)
    with pytest.raises(ValueError, match="fewer than max_rank"):
        evaluate_rank(d, np.zeros(6, int), gp2, qc2, gc2, max_rank=5)


def test_one_shot_c_entry_point():
    """ieee_eval_market1501: the single call a C host would make."""
    s = make_retrieval_set(50, 400, 10, 3, dim=64, sigma=2.0, seed=2)
    d = R.compute_distance_matrix(s.qf, s.gf).numpy()
    cmc_o, map_o = R.evaluate_rank(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, max_rank=10)
    lib = _lib.load()
    dev = torch.device("cuda")
    dd = torch.from_numpy(d).to(dev)
    lab = [torch.from_numpy(x).to(dev) for x in (s.q_pids, s.g_pids, s.q_camids, s.g_camids)]
    cap = 128
    nbytes = lib.ieee_eval_workspace_bytes(50, 400, cap)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    cmc = torch.empty(10, dtype=torch.float32, device=dev)
    summ = torch.empty(64, dtype=torch.uint8, device=dev)
    _lib.call("ieee_eval_market1501", dd.data_ptr(), 400, 50, 400, lab[0].data_ptr(), lab[1].data_ptr(),
              lab[2].data_ptr(), lab[3].data_ptr(), 10, cap, cmc.data_ptr(), summ.data_ptr(), ws.data_ptr(), nbytes,
              _lib.stream())
    res = _lib.EvalSummary.from_buffer_copy(summ.cpu().numpy().tobytes())
    assert np.array_equal(cmc.cpu().numpy(), cmc_o) and abs(res.mAP - map_o) < 1e-9 and res.status == 0
    rc = lib.ieee_eval_market1501(dd.data_ptr(), 400, 50, 400, lab[0].data_ptr(), lab[1].data_ptr(), lab[2].data_ptr(),
                                  lab[3].data_ptr(), 10, 2, cmc.data_ptr(), summ.data_ptr(), ws.data_ptr(), nbytes,
                                  _lib.stream())
    assert rc == _lib.ERR_CAPACITY


def test_one_call_retrieval_c_entry_point():
    """ieee_retrieve_eval: raw features + labels in, (cmc, summary, distance block) out, one C call."""
    s = make_retrieval_set(70, 500, 12, 3, dim=96, sigma=2.0, seed=5)
    lib = _lib.load()
    dev = torch.device("cuda")
    qf, gf = s.qf.to(dev), s.gf.to(dev)
    lab = [torch.from_numpy(x).to(dev) for x in (s.q_pids, s.g_pids, s.q_camids, s.g_camids)]
    Q, G, D, K = 70, 500, 96, 10
    nbytes = lib.ieee_retrieve_workspace_bytes(Q, G, D, 0, 0)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dist = torch.empty((Q, 512), dtype=torch.float32, device=dev)
    cmc = torch.empty(K, dtype=torch.float32, device=dev)
    summ = torch.empty(64, dtype=torch.uint8, device=dev)
    ap = torch.empty(Q, dtype=torch.float64, device=dev)

    def run(cap, cap_out):
        _lib.call("ieee_retrieve_eval", qf.data_ptr(), D, gf.data_ptr(), D, 0, Q, G, D, 0, 0, 0, lab[0].data_ptr(),
                  lab[1].data_ptr(), lab[2].data_ptr(), lab[3].data_ptr(), K, cap, cap_out, dist.data_ptr(), 512,
                  cmc.data_ptr(), summ.data_ptr(), ap.data_ptr(), None, ws.data_ptr(), nbytes, _lib.stream())
        return _lib.EvalSummary.from_buffer_copy(summ.cpu().numpy().tobytes())

    import ctypes
    need = ctypes.c_int32(0)
    res = run(0, ctypes.byref(need))                                       # sizing call: queries the capacity
    d = dist[:, :G].cpu().numpy()
    assert np.allclose(d, R.compute_distance_matrix(s.qf, s.gf).numpy(), rtol=1e-4, atol=1e-2)
    cmc_o, map_o = R.evaluate_rank(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, max_rank=K)
    pos = R.kept_positions(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    assert np.array_equal(cmc.cpu().numpy(), cmc_o) and abs(res.mAP - map_o) < 1e-9 and res.status == 0
    assert res.list_overflow == 0 and need.value >= max(p.size for p in pos)
    assert abs(res.mINP - R.mean_inverse_negative_penalty(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)) < 1e-12
    ap_o = np.array([((np.arange(p.size) + 1.0) / (p + 1.0)).sum() / p.size if p.size else 0.0 for p in pos])
    assert np.abs(ap.cpu().numpy() - ap_o).max() < 1e-12
    res2 = run(need.value, None)                                           # hinted call: asynchronous, same result
    assert res2.mAP == res.mAP and res2.list_overflow == 0
    res3 = run(2, None)                                                    # hint too small: flagged, not trusted
    assert 2 < res3.list_overflow <= need.value


@pytest.mark.parametrize("k", [1, 20, 21, 100])
def test_topk_ranked_list(k):
    s = make_retrieval_set(60, 2500, 20, 4, dim=64, sigma=2.0, seed=k)
    d = R.compute_distance_matrix(s.qf, s.gf).numpy()
    d[:, ::5] = np.round(d[:, ::5])                                        # inject ties
    idx_o, val_o = R.topk_kept(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, k)
    idx, val = topk_ranked_list(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, k=k)
    assert np.array_equal(idx.cpu().numpy(), idx_o) and np.array_equal(val.cpu().numpy(), val_o)
    # unmasked variant == plain stable argsort prefix (rerank.py:48)
    idx_u, _ = topk_ranked_list(d, k=k)
    assert np.array_equal(idx_u.cpu().numpy(), np.argsort(d, axis=1, kind="stable")[:, :k])


def test_topk_fewer_kept_than_k():
    d = np.arange(12, dtype=np.float32).reshape(2, 6)
    idx, val = topk_ranked_list(d, [1, 2], [1, 1, 1, 2, 2, 3], [0, 0], [0, 0, 1, 0, 1, 1], k=6)
    assert idx.cpu().tolist() == [[2, 3, 4, 5, -1, -1], [0, 1, 2, 4, 5, -1]]
    assert np.isinf(val.cpu().numpy()[0, 4:]).all()


def test_market1501_shape_full_size():
    """Config C2 at full size: 3368 x 15913, euclidean; oracle fed the SAME distmat bits."""
    s = market1501_shaped()
    from ieee_b200.metrics import compute_distance_matrix
    d_dev = compute_distance_matrix(s.qf.cuda(), s.gf.cuda())
    d = d_dev.cpu().numpy()
    cmc_o, map_o = R.evaluate_rank(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    cmc, mAP = evaluate_rank(d_dev, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    assert np.array_equal(cmc, cmc_o) and abs(mAP - map_o) < 1e-9 and 0.05 < mAP < 0.95


def test_cuhk03_protocol_matches_reference_for_fixed_seeds(golden_dir):
    """Single-gallery-shot protocol (rank.py:24-100, rank_cy.pyx:37-153): ranked lists from the GPU, sampling with
    NumPy's generator in the reference's call order -- equal to the golden file the compiled reference wrote, per seed."""
    from ieee_b200.metrics import rank as M
    g = np.load(os.path.join(golden_dir, "cuhk03_small.npz"))
    args = (g["distmat"], g["q_pids"], g["g_pids"], g["q_camids"], g["g_camids"])
    for seed in (0, 1234):
        for k in (5, 20):
            np.random.seed(seed)
            cmc, mAP = M.eval_cuhk03(*args, k)
            np.random.seed(seed)
            cmc_o, map_o = R.eval_cuhk03(*args, k)
            assert np.array_equal(cmc, cmc_o) and mAP == map_o                  # the oracle restatement, bit for bit
            np.testing.assert_allclose(cmc, g[f"cmc_s{seed}_k{k}"], rtol=0, atol=2e-7)   # rank_cy accumulates in float32
            assert abs(mAP - float(g[f"mAP_s{seed}_k{k}"])) < 1e-7
    # the fork's time ids (rank.py:48): one shared time id changes nothing; per-item time ids un-junk every pair
    np.random.seed(5)
    a = M.eval_cuhk03(*args, 20, q_timeids=np.zeros(60, int), g_timeids=np.zeros(400, int))
    np.random.seed(5)
    b = M.eval_cuhk03(*args, 20)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]
    np.random.seed(5)
    c = M.eval_cuhk03(*args, 20, q_timeids=np.arange(60), g_timeids=1000 + np.arange(400))
    np.random.seed(5)
    c_o = R.eval_cuhk03(*args, 20, q_timeids=np.arange(60), g_timeids=1000 + np.arange(400))
    assert np.array_equal(c[0], c_o[0]) and c[1] == c_o[1]
    # drop-in default: the fork's branch raises TypeError (rank.py:236-239); the protocol is an explicit opt-in
    with pytest.raises(TypeError):
        evaluate_rank(*args, max_rank=20, use_metric_cuhk03=True)
    M.ENABLE_CUHK03 = True
    try:
        np.random.seed(0)
        cmc, mAP = evaluate_rank(*args, max_rank=20, use_metric_cuhk03=True)
        np.testing.assert_allclose(cmc, g["cmc_s0_k20"], rtol=0, atol=2e-7)
    finally:
        M.ENABLE_CUHK03 = False
    with pytest.raises(ValueError):
        M.eval_cuhk03(np.zeros((2, 2000), np.float32), np.zeros(2, int), np.zeros(2000, int), np.zeros(2, int), np.ones(2000, int), 5)


def test_float64_distmat_is_ranked_in_float64_order():
    """evaluate_py (rank.py:117) argsorts the matrix in the dtype it arrives in.  Distances that only differ below
    float32 resolution are ordered there; a float32 copy ties them and the index rule can pick the other order."""
    rng = np.random.RandomState(3)
    Q, G = 40, 600
    d = rng.uniform(1.0, 2.0, size=(Q, G))
    q_pids, g_pids = rng.randint(0, 15, Q), rng.randint(0, 15, G)
    q_cams, g_cams = rng.randint(0, 3, Q), rng.randint(0, 3, G)
    # for every query: a relevant item and an irrelevant one at a LOWER index, equal in float32, relevant one closer in float64
    flips = 0
    for q in range(Q):
        rel = np.nonzero((g_pids == q_pids[q]) & (g_cams != q_cams[q]))[0]
        irr = np.nonzero(g_pids != q_pids[q])[0]
        if rel.size == 0 or irr.size == 0 or irr[0] > rel[-1]:
            continue
        r, w = rel[-1], irr[0]                                # w < r
        base = np.float64(np.float32(1.0 + 1e-3 * q))
        d[q, r], d[q, w] = base, base + 2e-9                  # equal after rounding to float32
        assert np.float32(d[q, r]) == np.float32(d[q, w]) and d[q, r] < d[q, w]
        flips += 1
    assert flips > 20
    cmc, mAP = evaluate_rank(d, q_pids, g_pids, q_cams, g_cams, max_rank=20)
    cmc_o, map_o = R.evaluate_rank(d, q_pids, g_pids, q_cams, g_cams, max_rank=20)       # float64 argsort, no ties
    assert np.array_equal(cmc, cmc_o) and abs(mAP - map_o) < 1e-12
    if ref.available():
        cmc_r, map_r = ref.evaluate_rank(d, q_pids, g_pids, q_cams, g_cams, max_rank=20)  # the reference's own evaluate_py
        assert np.array_equal(cmc, cmc_r) and abs(mAP - map_r) < 1e-12
    # the float32 copy really is a different problem: index order puts the irrelevant item first
    cmc32, map32 = evaluate_rank(d.astype(np.float32), q_pids, g_pids, q_cams, g_cams, max_rank=20)
    assert map32 < mAP
    # torch float64 tensors on the device take the same path
    cmc_t, map_t = evaluate_rank(torch.from_numpy(d).cuda(), q_pids, g_pids, q_cams, g_cams, max_rank=20)
    assert np.array_equal(cmc_t, cmc) and map_t == mAP
    # NaN last, -0 == +0, ties by index: same conventions as the float32 kernels
    d2 = np.round(rng.uniform(0, 8, size=(Q, G)))
    d2[:, ::17] = np.nan
    d2[:, 5] = -0.0
    cmc2, map2 = evaluate_rank(d2, q_pids, g_pids, q_cams, g_cams, max_rank=20)
    cmc2_o, map2_o = R.evaluate_rank(d2, q_pids, g_pids, q_cams, g_cams, max_rank=20)
    assert np.array_equal(cmc2, cmc2_o) and abs(map2 - map2_o) < 1e-12


def test_limits_are_reported_in_python():
    d = np.zeros((3, 10), np.float32)
    lab = (np.zeros(3, int), np.zeros(10, int), np.zeros(3, int), np.ones(10, int))
    with pytest.raises(ValueError, match="ranked lists hold"):
        topk_ranked_list(d, *lab, k=5000)
    big = np.zeros((2, 9000), np.float32)
    with pytest.raises(ValueError, match="max_rank"):
        evaluate_rank(big, np.zeros(2, int), np.zeros(9000, int), np.zeros(2, int), np.ones(9000, int), max_rank=9000)
