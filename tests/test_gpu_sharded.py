"""GPU parity of the gallery-sharded path: the kernels' shard arguments on one GPU, and -- when the box has two
GPUs -- the real thing over NCCL (one process per GPU)."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import restatement as R
from ieee_b200 import _lib
from ieee_b200.engine import RetrievalEvaluator, shard_bounds
from ieee_b200.metrics.rank import GalleryLabels, RankStages, topk_ranked_list
from ieee_b200.testing import make_retrieval_set

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shards", [2, 3, 8])
def test_shard_stages_on_one_gpu(shards):
    """gather / count per shard with global offsets, lists concatenated as the all-gather would, counts summed as the
    all-reduce would: bit-identical to the unsharded evaluation."""
    s = make_retrieval_set(150, 1203, 20, 4, dim=64, sigma=2.0, seed=shards)
    d = R.compute_distance_matrix(s.qf, s.gf).numpy()
    d[:, ::3] = np.round(d[:, ::3])                                  # ties, also across shard boundaries
    cmc_o, map_o, info = R.eval_market1501(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, 20, return_info=True)
    dev = torch.device("cuda")
    Q, G = d.shape
    qp, qc = torch.from_numpy(s.q_pids).to(dev), torch.from_numpy(s.q_camids).to(dev)
    parts = []
    for r in range(shards):
        g0, g1 = shard_bounds(G, shards, r)
        dl = torch.from_numpy(np.ascontiguousarray(d[:, g0:g1])).to(dev)
        parts.append((g0, g1, dl, GalleryLabels(s.g_pids[g0:g1], s.g_camids[g0:g1], dev)))
    cap = max(p[3].list_cap(qp) for p in parts)

    def run(width):
        stages = [RankStages(Q, cap, shards, dev, width) for _ in parts]
        for st, (g0, g1, dl, gal) in zip(stages, parts):
            st.gather(dl, qp, qc, gal, g0)
        rel_all = torch.stack([st.rel for st in stages]).contiguous()          # what the all-gather produces
        for st, (g0, g1, dl, gal) in zip(stages, parts):
            st.count(dl, g1 - g0, g0, rel_all)
        total = torch.stack([st.counts for st in stages]).sum(0).to(torch.int32).contiguous()
        ties = torch.stack([st.flags[1:2] for st in stages]).sum(0).contiguous()
        longest = int(torch.stack([st.flags[2] for st in stages]).max().item())
        fin = stages[0]
        fin.finalize(G, 20, counts=total, ties=ties)
        return fin, fin.read_summary(), longest

    fin, summary, longest = run(0)                                           # rows as wide as shards * cap
    assert np.array_equal(fin.cmc.cpu().numpy(), cmc_o) and abs(summary.mAP - map_o) < 1e-9
    assert np.array_equal(fin.first.cpu().numpy(), info["first_hit"])
    pos = R.kept_positions(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    assert longest == max(p.size for p in pos) <= shards * cap
    fin2, summary2, longest2 = run(longest)                                  # rows as wide as the longest merged list
    assert longest2 == longest and fin2.counts.shape[1] == longest + 2
    assert np.array_equal(fin2.cmc.cpu().numpy(), cmc_o) and summary2.mAP == summary.mAP
    assert np.array_equal(fin2.first.cpu().numpy(), info["first_hit"])
    if longest > 1:
        _, _, longest3 = run(longest - 1)                                    # too narrow: reported, never silent
        assert longest3 == longest


def test_topk_merge_across_shards():
    s = make_retrieval_set(64, 1000, 16, 3, dim=64, sigma=2.0, seed=1)
    d = R.compute_distance_matrix(s.qf, s.gf).numpy()
    d[:, ::4] = np.round(d[:, ::4])
    k, shards = 20, 4
    idx_o, val_o = R.topk_kept(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, k)
    idx_parts, val_parts = [], []
    for r in range(shards):
        g0, g1 = shard_bounds(d.shape[1], shards, r)
        i, v = topk_ranked_list(np.ascontiguousarray(d[:, g0:g1]), s.q_pids, s.g_pids[g0:g1], s.q_camids, s.g_camids[g0:g1],
                                k=k, g_offset=g0)
        idx_parts.append(i)
        val_parts.append(v)
    idx_all, val_all = torch.stack(idx_parts).contiguous(), torch.stack(val_parts).contiguous()
    idx = torch.empty_like(idx_parts[0])
    val = torch.empty_like(val_parts[0])
    _lib.call("ieee_topk_merge", idx_all.data_ptr(), val_all.data_ptr(), shards, d.shape[0], k, idx.data_ptr(), val.data_ptr(),
              _lib.stream())
    assert np.array_equal(idx.cpu().numpy(), idx_o) and np.array_equal(val.cpu().numpy(), val_o)


@pytest.mark.parametrize("shards", [1, 2, 3])
def test_peer_exchange_protocol_on_one_gpu(shards):
    """The peer-memory exchange (ieee_rank_*_peer) with `shards` virtual ranks on ONE device: one buffer and one stream
    per virtual rank, kernels of different ranks handing over through the flag words exactly as they do across GPUs.
    Two query blocks of different size, so that epochs, block offsets and the count-table slots are all exercised."""
    import ctypes as C
    from ieee_b200.peer import LocalPeers
    s = make_retrieval_set(150, 1203, 20, 4, dim=64, sigma=2.0, seed=40 + shards)
    d = R.compute_distance_matrix(s.qf, s.gf).numpy()
    d[:, ::3] = np.round(d[:, ::3])                                  # ties, also across shard boundaries
    cmc_o, map_o, info = R.eval_market1501(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, 20, return_info=True)
    pos = R.kept_positions(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    dev = torch.device("cuda")
    lib = _lib.load()
    Q, G = d.shape
    qp, qc = torch.from_numpy(s.q_pids).to(dev), torch.from_numpy(s.q_camids).to(dev)
    parts = []
    for r in range(shards):
        g0, g1 = shard_bounds(G, shards, r)
        dl = torch.from_numpy(np.ascontiguousarray(d[:, g0:g1])).to(dev)
        parts.append((g0, g1, dl, GalleryLabels(s.g_pids[g0:g1], s.g_camids[g0:g1], dev)))
    cap = max(p[3].list_cap(qp) for p in parts)
    W = min(shards * cap, max(p.size for p in pos))
    Qb_max = 96
    peers = LocalPeers(shards, dev, lib.ieee_peer_exchange_bytes(Qb_max, Q, cap, W, shards))
    streams = [torch.cuda.Stream() for _ in range(shards)]
    stats = [torch.zeros(4, dtype=torch.int64, device=dev) for _ in range(shards)]
    keep = []
    results = [(torch.empty(20, dtype=torch.float32, device=dev), torch.empty(64, dtype=torch.uint8, device=dev),
                torch.zeros(4, dtype=torch.int64, device=dev)) for _ in range(shards)]
    torch.cuda.synchronize()
    epoch = 0
    for q0 in range(0, Q, Qb_max):
        q1 = min(Q, q0 + Qb_max)
        Qb = q1 - q0
        epoch += 1
        for r, (g0, g1, dl, gal) in enumerate(parts):
            ex = peers.descriptor(r, Qb_max, Qb, Q, q0, cap, W, epoch)
            junk = torch.empty((Qb, cap), dtype=torch.int64, device=dev)
            n_rel, n_junk = torch.empty(Qb, dtype=torch.int32, device=dev), torch.empty(Qb, dtype=torch.int32, device=dev)
            keep.append((junk, n_rel, n_junk))
            blk = dl[q0:q1]
            with torch.cuda.stream(streams[r]):
                st = streams[r].cuda_stream
                _lib.call("ieee_rank_gather_peer", blk.data_ptr(), blk.stride(0), g1 - g0, qp[q0:q1].data_ptr(), qc[q0:q1].data_ptr(),
                          gal.camids.data_ptr(), gal.group.data_ptr(), g0, n_rel.data_ptr(), junk.data_ptr(), n_junk.data_ptr(),
                          stats[r].data_ptr(), C.byref(ex), st)
                _lib.call("ieee_rank_count_peer", blk.data_ptr(), blk.stride(0), g1 - g0, g0, n_rel.data_ptr(), junk.data_ptr(),
                          n_junk.data_ptr(), stats[r].data_ptr(), C.byref(ex), st)
                # the metrics kernel of the last block also reduces over all Q queries
                cmc, summ, st_out = results[r]
                _lib.call("ieee_rank_metrics_peer", G, 20, stats[r].data_ptr(), cmc.data_ptr(), summ.data_ptr(),
                          st_out.data_ptr(), C.byref(ex), st)
    torch.cuda.synchronize()
    off_ap, off_first = (lib.ieee_peer_result_offset(i, Qb_max, Q, cap, W, shards) for i in (0, 1))
    ap_o = np.array([((np.arange(p.size) + 1.0) / (p + 1.0)).sum() / p.size if p.size else 0.0 for p in pos])
    for r, (cmc, summ, st_out) in enumerate(results):
        summary = _lib.EvalSummary.from_buffer_copy(summ.cpu().numpy().tobytes())
        assert np.array_equal(cmc.cpu().numpy(), cmc_o) and abs(summary.mAP - map_o) < 1e-9 and summary.list_overflow == 0
        over, ties, longest = st_out.cpu().numpy()[:3]
        assert over == 0 and longest == max(p.size for p in pos) and summary.num_ties == ties
        ap = peers.views[r][off_ap: off_ap + 8 * Q].view(torch.float64).cpu().numpy()
        first = peers.views[r][off_first: off_first + 4 * Q].view(torch.int32).cpu().numpy()
        assert np.abs(ap - ap_o).max() < 1e-12 and np.array_equal(first, info["first_hit"])
    assert all(results[0][1].cpu().numpy().tobytes() == x[1].cpu().numpy().tobytes() for x in results)   # bit-identical
    peers.free()


def _tied_set():
    """Gallery with rows duplicated ACROSS the two shards: bit-equal distances on different ranks, so the merged order
    depends on the global-index tie rule."""
    s = make_retrieval_set(300, 2001, 30, 4, dim=256, sigma=2.5, seed=23, distractor_frac=0.1)
    gf = s.gf.clone()
    g_pids, g_camids = s.g_pids.copy(), s.g_camids.copy()
    src = np.arange(0, 400, 2)
    dst = 2001 - 1 - src                                # second shard (rows >= 1001)
    gf[dst] = gf[src]
    g_pids[dst], g_camids[dst] = g_pids[src], (g_camids[src] + 1) % 4
    return s, gf, g_pids, g_camids


def _ranked_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    s, gf, g_pids, g_camids = _tied_set()
    G = gf.shape[0]
    g0, g1 = shard_bounds(G, world, rank)
    ev = RetrievalEvaluator(gf[g0:g1].cuda(), g_pids[g0:g1], g_camids[g0:g1], group=dist.group.WORLD, g_offset=g0, g_total=G)
    cmc, mAP, info = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True)
    idx, val = ev.ranked_lists(s.qf.cuda(), s.q_pids, s.q_camids, k=25)
    idx_u, _ = ev.ranked_lists(s.qf.cuda(), k=7)        # unmasked
    gathered = [torch.empty((300, shard_bounds(G, world, r)[1] - shard_bounds(G, world, r)[0]), device="cuda") for r in range(world)]
    dist.all_gather(gathered, info["distmat"].contiguous())
    if rank == 0:
        out["idx"], out["val"], out["idx_u"] = idx.cpu().numpy(), val.cpu().numpy(), idx_u.cpu().numpy()
        out["d"] = torch.cat(gathered, 1).cpu().numpy()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_ranked_lists():
    """north_star: local top-k per gallery slice, all-gather over NVLink, merge -- bit-exact incl. ties across shards."""
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = mp.Manager().dict()
    mp.spawn(_ranked_worker, args=(2, port, out), nprocs=2, join=True)
    s, gf, g_pids, g_camids = _tied_set()
    d = out["d"]
    assert (d[:, 0] == d[:, 2000]).all()                                   # the duplicates really tie across the shards
    idx_o, val_o = R.topk_kept(d, s.q_pids, g_pids, s.q_camids, g_camids, 25)
    assert np.array_equal(out["idx"], idx_o) and np.array_equal(out["val"], val_o)
    none = np.full(300, -1)
    idx_uo, _ = R.topk_kept(d, none, g_pids, none - 1, g_camids, 7)
    assert np.array_equal(out["idx_u"], idx_uo)


def test_ranked_lists_on_one_gpu(tmp_path):
    s, gf, g_pids, g_camids = _tied_set()
    ev = RetrievalEvaluator(gf.cuda(), g_pids, g_camids, block_bytes=128 * 2001 * 4)      # several query blocks
    _, _, info = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True)
    d = info["distmat"].cpu().numpy()
    idx, val = ev.ranked_lists(s.qf, s.q_pids, s.q_camids, k=25)                           # host queries are copied
    idx_o, val_o = R.topk_kept(d, s.q_pids, g_pids, s.q_camids, g_camids, 25)
    assert np.array_equal(idx.cpu().numpy(), idx_o) and np.array_equal(val.cpu().numpy(), val_o)
    # the consumer takes the lists instead of a Q x G matrix (reidtools.py:49,109-145)
    from ieee_b200.utils.reidtools import ranked_lists
    dataset = ([("q%d.jpg" % i, int(p), int(c)) for i, (p, c) in enumerate(zip(s.q_pids, s.q_camids))],
               [("g%d.jpg" % i, int(p), int(c)) for i, (p, c) in enumerate(zip(g_pids, g_camids))])
    a = ranked_lists(d, dataset, topk=10)
    b = ranked_lists(None, dataset, topk=10, ranked=(idx, val))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def _nccl_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    s = make_retrieval_set(500, 3001, 40, 4, dim=256, sigma=2.5, seed=17, distractor_frac=0.1)
    g0, g1 = shard_bounds(3001, world, rank)
    ev = RetrievalEvaluator(s.gf[g0:g1].cuda(), s.g_pids[g0:g1], s.g_camids[g0:g1], group=dist.group.WORLD, g_offset=g0,
                            g_total=3001, block_bytes=256 * (g1 - g0) * 4)                     # two query blocks
    assert ev.exchange == "peer"
    cmc, mAP, info = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids, return_distmat=True)
    # the NCCL exchange (all-gather + all-reduce launches) and the peer-memory exchange agree to the last bit,
    # twice in a row (second time: capacity memo hit, narrower count rows, next epochs)
    ev_n = RetrievalEvaluator(s.gf[g0:g1].cuda(), s.g_pids[g0:g1], s.g_camids[g0:g1], group=dist.group.WORLD, g_offset=g0,
                              g_total=3001, exchange="nccl", center=ev.center)
    for _ in range(2):
        c_n, m_n, i_n = ev_n.evaluate(s.qf.cuda(), s.q_pids, s.q_camids)
        c_p, m_p, i_p = ev.evaluate(s.qf.cuda(), s.q_pids, s.q_camids)
        assert np.array_equal(c_n, c_p) and m_n == m_p and i_n["num_ties"] == i_p["num_ties"] and i_n["mINP"] == i_p["mINP"]
        assert torch.equal(i_n["ap"], i_p["ap"]) and torch.equal(i_n["first"], i_p["first"])
    assert np.array_equal(c_p, cmc) and m_p == mAP
    gathered = [torch.empty((500, shard_bounds(3001, world, r)[1] - shard_bounds(3001, world, r)[0]), device="cuda") for r in range(world)]
    dist.all_gather(gathered, info["distmat"].contiguous())
    if rank == 0:
        out["cmc"], out["mAP"], out["d"] = cmc, mAP, torch.cat(gathered, 1).cpu().numpy()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_nccl_evaluation():
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, port, out), nprocs=2, join=True)
    s = make_retrieval_set(500, 3001, 40, 4, dim=256, sigma=2.5, seed=17, distractor_frac=0.1)
    cmc_o, map_o = R.evaluate_rank(out["d"], s.q_pids, s.g_pids, s.q_camids, s.g_camids)
    assert np.array_equal(out["cmc"], cmc_o) and abs(out["mAP"] - map_o) < 1e-9


def _peer_one_call_worker(rank, world, port, out):
    import torch.distributed as dist
    from ieee_b200 import engine
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    s = make_retrieval_set(500, 3001, 40, 4, dim=256, sigma=2.5, seed=17, distractor_frac=0.1)
    g0, g1 = shard_bounds(3001, world, rank)
    # label tensors (the capacity memo is keyed on tensor identity) and one query block (default block budget)
    qp, qc = torch.from_numpy(s.q_pids).to(dev), torch.from_numpy(s.q_camids).to(dev)
    gp, gc = torch.from_numpy(s.g_pids[g0:g1]).to(dev), torch.from_numpy(s.g_camids[g0:g1]).to(dev)
    qf = s.qf.to(dev)
    ev = RetrievalEvaluator(s.gf[g0:g1].to(dev), gp, gc, group=dist.group.WORLD, g_offset=g0, g_total=3001)
    assert ev.exchange == "peer"
    calls, real_call = [], _lib.call

    def spy(name, *args):
        calls.append(name)
        return real_call(name, *args)

    def run(evaluator):
        calls.clear()
        cmc, mAP, info = evaluator.evaluate(qf, qp, qc)
        return (cmc, mAP, info["ap"], info["first"], info["mINP"], info["num_ties"]), list(calls)

    def same(a, b):
        assert np.array_equal(a[0], b[0]) and a[1] == b[1] and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
        assert a[4] == b[4] and a[5] == b[5]

    _lib.call = spy
    try:
        staged, c1 = run(ev)                                  # sizes unknown: the staged loop with the peer exchange
        assert "ieee_rank_gather_peer" in c1 and "ieee_retrieve_eval_prepared_peer" not in c1
        key = [k for k in engine._CAP_MEMO if k[0] == ev._label_keys][0]
        assert engine._CAP_MEMO[key][1] > 0                   # the row width is memoised
        hit, c2 = run(ev)                                     # memo hit: the whole step in one call
        assert "ieee_retrieve_eval_prepared_peer" in c2 and "ieee_rank_gather_peer" not in c2
        same(staged, hit)
        ev_n = RetrievalEvaluator(s.gf[g0:g1].to(dev), gp, gc, group=dist.group.WORLD, g_offset=g0, g_total=3001,
                                  exchange="nccl", center=ev.center)
        same(hit, run(ev_n)[0])
        engine._CAP_MEMO[key] = (2, 0)          # capacity far too small, no width: the staged route overflows, runs again
        poisoned, c3 = run(ev)
        assert "ieee_retrieve_eval_prepared_peer" not in c3
        same(hit, poisoned)
        engine._CAP_MEMO[key] = (2, 1)          # with a width: the one call overflows and the staged route runs exactly
        fallback, c4 = run(ev)
        assert "ieee_retrieve_eval_prepared_peer" in c4 and "ieee_rank_gather_peer" in c4
        same(hit, fallback)
    finally:
        _lib.call = real_call
    out[rank] = True
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_peer_one_call_evaluation():
    """The memoised one-call step of a sharded gallery (ieee_retrieve_eval_prepared_peer) against the staged peer loop
    and the NCCL exchange, bit for bit, and its overflow fall-back to the staged loop."""
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = mp.Manager().dict()
    mp.spawn(_peer_one_call_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: True, 1: True}
