"""RetrievalEvaluator.capture(): one query block's evaluation as a CUDA graph.  Replays equal evaluate() bit for bit,
run no foreign call and no synchronisation, recover from lists that outgrow the captured sizes, and -- over a sharded
gallery -- keep the peer exchange's epoch on the device (ieee_retrieve_eval_prepared_peer_dev_epoch)."""
import os
import socket

import numpy as np
import pytest
import torch

from ieee_b200 import _lib, engine
from ieee_b200.engine import RetrievalEvaluator, feature_center, shard_bounds
from ieee_b200.testing import make_retrieval_set

pytestmark = pytest.mark.gpu

Q, G = 300, 1700


def _sets(seed=3, **kw):
    """Three query sets of Q rows against one gallery of G rows."""
    return make_retrieval_set(3 * Q, G, 40, 4, dim=256, sigma=2.5, seed=seed, distractor_frac=0.1, **kw)


def _queries(s, i, dev, dtype=torch.float32):
    sl = slice(i * Q, (i + 1) * Q)
    return (s.qf[sl].to(dev, dtype), torch.from_numpy(s.q_pids[sl]).to(dev), torch.from_numpy(s.q_camids[sl]).to(dev))


def _same(a, b, distmat=False):
    (c1, m1, i1), (c2, m2, i2) = a, b
    assert np.array_equal(c1, c2) and m1 == m2 and i1["mINP"] == i2["mINP"]
    assert i1["num_valid"] == i2["num_valid"] and i1["num_ties"] == i2["num_ties"]
    assert torch.equal(i1["ap"], i2["ap"]) and torch.equal(i1["first"], i2["first"])
    if distmat:
        assert torch.equal(i1["distmat"], i2["distmat"])


@pytest.mark.parametrize("metric,normalize,dtype", [("euclidean", False, torch.float32), ("cosine", True, torch.float32),
                                                    ("euclidean", False, torch.bfloat16)])
def test_replay_equals_evaluate(metric, normalize, dtype):
    """f16x3 euclidean, cosine on normalised rows, and the 1-pass bf16 mode: three query contents copied into the
    static inputs, each replay bit for bit what evaluate() of the same evaluator returns on the same contents."""
    dev = torch.device("cuda")
    s = _sets()
    ev = RetrievalEvaluator(s.gf.to(dev, dtype), s.g_pids, s.g_camids, metric, normalize)
    h = ev.capture(*_queries(s, 0, dev, dtype), return_distmat=True)
    assert h.qf.dtype == dtype and h.qf.shape == (Q, 256) and h.q_pids.dtype == torch.int64
    for i in (1, 2, 0):
        qf, qp, qc = _queries(s, i, dev, dtype)
        h.qf.copy_(qf)
        h.q_pids.copy_(qp)
        h.q_camids.copy_(qc)
        got = h.replay()
        assert set(got[2]) == {"ap", "first", "mINP", "num_valid", "num_ties", "cap", "distmat"}
        _same(got, ev.evaluate(qf, qp, qc, return_distmat=True), distmat=True)


def test_replay_runs_no_library_call_and_launch_does_not_wait(monkeypatch):
    dev = torch.device("cuda")
    s = _sets(seed=4)
    ev = RetrievalEvaluator(s.gf.to(dev), s.g_pids, s.g_camids)
    h = ev.capture(*_queries(s, 0, dev))
    ref = ev.evaluate(*_queries(s, 0, dev))
    calls, waits = [], []
    real_call = _lib.call
    monkeypatch.setattr(_lib, "call", lambda name, *a: (calls.append(name), real_call(name, *a))[1])
    got = h.replay()
    assert calls == []
    _same(got, ref)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: waits.append("device"))
    monkeypatch.setattr(torch.cuda.Stream, "synchronize", lambda *a, **k: waits.append("stream"))
    h.launch()
    assert calls == [] and waits == []
    monkeypatch.undo()
    _same(h.result(), ref)


def test_overflow_recaptures_with_exact_sizes():
    """A planted capacity that is too small is corrected by capture()'s evaluate(); labels that need more than the
    captured capacity are flagged by the replay, which captures again with exact sizes and returns the right numbers."""
    dev = torch.device("cuda")
    s = _sets(seed=5)
    g_pids = s.g_pids.copy()
    g_pids[:300] = 7                                  # identity 7: a group far larger than any other
    gp, gc = torch.from_numpy(g_pids).to(dev), torch.from_numpy(s.g_camids).to(dev)
    ev = RetrievalEvaluator(s.gf.to(dev), gp, gc)
    qf, qp, qc = _queries(s, 0, dev)
    small = torch.where(qp == 7, torch.full_like(qp, 8), qp)
    engine._CAP_MEMO[ev._memo_key(small)] = (1, 0)
    h = ev.capture(qf, small, qc)
    cap_small = h.cap
    assert 1 < cap_small < 300
    _same(h.replay(), ev.evaluate(h.qf, h.q_pids, h.q_camids))
    big = qp.clone()
    big[:5] = 7
    h.q_pids.copy_(big)
    got = h.replay()
    assert h.cap >= 300 > cap_small and got[2]["cap"] == h.cap
    _same(got, ev.evaluate(qf, big, qc))


def test_unsupported_configurations_raise():
    dev = torch.device("cuda")
    s = _sets(seed=6)
    gf = s.gf.to(dev)
    q = _queries(s, 0, dev)
    for kw, what in (({"rerank": True}, "rerank=True"), ({"rerank": "gnn"}, "gnn")):
        with pytest.raises(ValueError, match=what):
            RetrievalEvaluator(gf, s.g_pids, s.g_camids, **kw).capture(*q)
    with pytest.raises(ValueError, match="from_host"):
        RetrievalEvaluator.from_host(s.gf.pin_memory(), s.g_pids, s.g_camids).capture(*q)
    with pytest.raises(ValueError, match="one query block"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, block_bytes=128 * G * 4).capture(*q)     # 128-row blocks
    lib = _lib.load()
    prev = lib.ieee_set_debug_flags(128)
    try:
        with pytest.raises(ValueError, match="timeline"):
            RetrievalEvaluator(gf, s.g_pids, s.g_camids).capture(*q)
    finally:
        lib.ieee_set_debug_flags(prev)


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _group_errors_worker(rank, world, port, backend, out):
    """gloo, two ranks sharing one GPU: a sharded gallery with the NCCL-launch exchange.  NCCL, one rank: a query_group."""
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    dist.init_process_group(backend, rank=rank, world_size=world, **({"device_id": dev} if backend == "nccl" else {}))
    s = _sets(seed=7)
    q = _queries(s, 0, dev)
    if backend == "gloo":
        g0, g1 = shard_bounds(G, world, rank)
        ev = RetrievalEvaluator(s.gf[g0:g1].to(dev), s.g_pids[g0:g1], s.g_camids[g0:g1], group=dist.group.WORLD,
                                g_offset=g0, g_total=G)
        assert ev.exchange == "nccl"
        with pytest.raises(ValueError, match="peer"):
            ev.capture(*q)
    else:
        ev = RetrievalEvaluator(s.gf.to(dev), s.g_pids, s.g_camids, rerank="gnn", query_group=dist.group.WORLD)
        with pytest.raises(ValueError, match="query_group"):
            ev.capture(*q)
    dist.barrier()
    out[rank] = True
    dist.destroy_process_group()


@pytest.mark.parametrize("backend,world", [("gloo", 2), ("nccl", 1)])
def test_unsupported_process_groups_raise(backend, world):
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_group_errors_worker, args=(world, _free_port(), backend, out), nprocs=world, join=True)
    assert dict(out) == {r: True for r in range(world)}


@pytest.mark.parametrize("shards", [2, 3])
def test_device_epoch_entry_with_virtual_ranks(shards):
    """ieee_retrieve_eval_prepared_peer_dev_epoch captured once per virtual rank (one exchange buffer and one stream per
    rank, all on one GPU), every rank's graph replayed for three query contents: each replay equals the host-epoch
    entry on the same inputs (cmc, summary, statistics, ap, first, distances), and each advances the epoch word by one."""
    from ieee_b200.peer import LocalPeers
    dev = torch.device("cuda")
    lib = _lib.load()
    s = _sets(seed=10 + shards)
    sets = [_queries(s, i, dev) for i in range(3)]
    center = feature_center(sets[0][0])
    evs = []
    for r in range(shards):
        g0, g1 = shard_bounds(G, shards, r)
        evs.append(RetrievalEvaluator(s.gf[g0:g1].to(dev), s.g_pids[g0:g1], s.g_camids[g0:g1], g_offset=g0, g_total=G,
                                      center=center))
    cap = max(ev.labels.list_cap(qp) for ev in evs for _, qp, _ in sets)
    W = shards * cap
    k_eff = 20
    nbytes = lib.ieee_peer_exchange_bytes(Q, Q, cap, W, shards)
    ws_bytes = lib.ieee_retrieve_prepared_peer_workspace_bytes(Q, 256, _lib.PRECISIONS["f16x3"], cap)
    streams = [torch.cuda.Stream() for _ in range(shards)]

    def buffers(ev):
        return {"ws": torch.empty(ws_bytes, dtype=torch.uint8, device=dev), "block": ev._new_block(Q),
                "res": torch.zeros(96 + 4 * k_eff, dtype=torch.uint8, device=dev),
                "ap": torch.empty(Q, dtype=torch.float64, device=dev), "first": torch.empty(Q, dtype=torch.int32, device=dev)}

    def launch(r, inputs, b, ex, epoch=None):
        evs[r]._one_call_launch(*inputs, cap, b["block"], b["ws"], b["res"], b["ap"], b["first"], None, ex, epoch)

    def on_every_rank(fn):
        cur = torch.cuda.current_stream()
        for r in range(shards):
            streams[r].wait_stream(cur)
            with torch.cuda.stream(streams[r]):
                fn(r)
        for st in streams:
            cur.wait_stream(st)
        torch.cuda.synchronize()

    graph_peers, host_peers = LocalPeers(shards, dev, nbytes), LocalPeers(shards, dev, nbytes)
    static = tuple(t.clone() for t in sets[0])
    mine = [buffers(ev) for ev in evs]
    host = [buffers(ev) for ev in evs]
    epochs = [torch.ones(1, dtype=torch.int64, device=dev) for _ in range(shards)]
    graphs = [torch.cuda.CUDAGraph() for _ in range(shards)]
    torch.cuda.synchronize()
    for r in range(shards):
        with torch.cuda.graph(graphs[r], stream=streams[r]):
            launch(r, static, mine[r], graph_peers.descriptor(r, Q, Q, Q, 0, cap, W, 0), epochs[r])
    try:
        for step, inputs in enumerate([sets[1], sets[2], sets[0], sets[1]]):
            for t, x in zip(static, inputs):
                t.copy_(x)
            on_every_rank(lambda r: graphs[r].replay())
            assert [int(e.item()) for e in epochs] == [step + 2] * shards
            on_every_rank(lambda r: launch(r, inputs, host[r], host_peers.descriptor(r, Q, Q, Q, 0, cap, W, step + 1)))
            for r in range(shards):
                a, b = mine[r], host[r]
                assert torch.equal(a["res"], b["res"]) and torch.equal(a["ap"], b["ap"]) and torch.equal(a["first"], b["first"])
                assert torch.equal(a["block"], b["block"])
                summary = _lib.EvalSummary.from_buffer_copy(a["res"][32:96].cpu().numpy().tobytes())
                assert summary.status == _lib.OK and summary.list_overflow == 0 and summary.num_valid > 0
            assert all(torch.equal(mine[0]["res"][32:], m["res"][32:]) for m in mine)     # the same cmc and summary
    finally:
        del graphs
        graph_peers.free()
        host_peers.free()


def _two_gpu_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    s = _sets(seed=12)
    g0, g1 = shard_bounds(G, world, rank)
    gp, gc = torch.from_numpy(s.g_pids[g0:g1]).to(dev), torch.from_numpy(s.g_camids[g0:g1]).to(dev)
    ev = RetrievalEvaluator(s.gf[g0:g1].to(dev), gp, gc, group=dist.group.WORLD, g_offset=g0, g_total=G)
    assert ev.exchange == "peer"
    h = ev.capture(*_queries(s, 0, dev), return_distmat=True)
    for i in (1, 2, 0, 1):
        qf, qp, qc = _queries(s, i, dev)
        h.qf.copy_(qf)
        h.q_pids.copy_(qp)
        h.q_camids.copy_(qc)
        _same(h.replay(), ev.evaluate(qf, qp, qc, return_distmat=True), distmat=True)
        assert int(h.epoch.item()) >= 2           # (a replay that captures again with larger sizes starts a new word)
    out[rank] = True
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_replay_equals_evaluate():
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_two_gpu_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert dict(out) == {0: True, 1: True}
