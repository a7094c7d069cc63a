"""GNN re-ranking shared by the ranks of a query_group (RetrievalEvaluator(rerank="gnn", query_group=...)): the library's
phases with virtual ranks on one GPU, the Python plumbing in a process group of one, and -- when the box has two GPUs --
the real thing over NCCL, all bit for bit against one GPU doing all the work."""
import ctypes as C
import functools
import os
import socket

import numpy as np
import pytest
import torch

from ieee_b200 import _lib
from ieee_b200.engine import PackedFeatures, RetrievalEvaluator, rerank_owned
from ieee_b200.testing import make_retrieval_set

pytestmark = pytest.mark.gpu
PHASES = ("ieee_gnn_stream_neighbours_rows", "ieee_gnn_stream_symbolic", "ieee_gnn_stream_sizes_sync", "ieee_gnn_stream_numeric",
          "ieee_gnn_stream_csc")


def r32(x):
    return (x + 31) // 32 * 32


def unit(t):
    return torch.nn.functional.normalize(t.float(), dim=1)


def counts_of(scratch, Q, G, k1, k2):
    off = (C.c_size_t * 10)()
    _lib.call("ieee_gnn_stream_layout", Q, G, k1, k2, None, off)
    return [scratch[off[i]: off[i] + 4 * (Q + G)].view(torch.int32) for i in range(4)]


def work_arrays(work, Q, G, k1, k2, sizes):
    off = (C.c_size_t * 10)()
    _lib.call("ieee_gnn_stream_layout", Q, G, k1, k2, sizes, off)
    n = (sizes[3], sizes[3], sizes[4], sizes[4], sizes[5], sizes[5])
    return [work[off[4 + i]: off[4 + i] + 4 * n[i]].view(torch.int32) for i in range(6)]


def run_virtual_ranks(s, world, k1, k2, dtype=torch.float32, normalize=False):
    """Each virtual rank runs every phase on its own rows (at its own strip width); between the phases the owned pieces
    are merged as the exchanges merge them (rows copied for the all-gathers, int32 sums for the rest).  Every merged
    structure and every rank's query rows equal the ungrouped evaluator's."""
    qf, gf = s.qf.cuda().to(dtype), s.gf.cuda().to(dtype)
    if not normalize:
        qf, gf = unit(qf).to(dtype), unit(gf).to(dtype)
    Q, G = qf.shape[0], gf.shape[0]
    N = Q + G
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, normalize_feature=normalize, rerank="gnn", k1=k1, k2=k2,
                            max_rank=min(20, G))
    _, _, info = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    ref, want = ev._rr, info["distmat"]
    qpk = PackedFeatures(qf, ev.metric, ev.normalize, ev.precision, None)
    gpk = ev.chunks[0][1]
    lib, dev, st = _lib.load(), qf.device, _lib.stream()
    # the reference counts: the one-GPU symbolic phase
    sc_ref = torch.empty(lib.ieee_gnn_stream_scratch_bytes(Q, G, k1, 0), dtype=torch.uint8, device=dev)
    sizes_ref = (C.c_int64 * 6)()
    _lib.call("ieee_gnn_stream_graph_bytes_sync", ref["rank"].data_ptr(), Q, G, k1, k2, sc_ref.data_ptr(), sc_ref.numel(),
              sizes_ref, st)
    ranks = []
    for r in range(world):
        budget = (256 * (1 + r % 3)) * 4 * (r32(N) + k1)
        sc = lib.ieee_gnn_stream_scratch_bytes(Q, G, k1, budget)
        ranks.append(dict(own=rerank_owned(Q, G, world, r), budget=budget, sc=torch.empty(sc, dtype=torch.uint8, device=dev),
                          rank=torch.full((N, k1), -7, dtype=torch.int32, device=dev),
                          S=torch.full((N, k1), float("nan"), device=dev)))

    def gather(get):
        full = get(ranks[0]).clone()
        for x in ranks:
            q0, q1, g0, g1 = x["own"]
            full[q0:q1] = get(x)[q0:q1]
            full[Q + g0: Q + g1] = get(x)[Q + g0: Q + g1]
        for x in ranks:
            get(x).copy_(full)
        return full

    def summed(get):
        full = functools.reduce(lambda a, b: a + b, [get(x) for x in ranks])
        for x in ranks:
            get(x).copy_(full)
        return full

    for x in ranks:
        _lib.call("ieee_gnn_stream_neighbours_rows", qpk.buf.data_ptr(), Q, gpk.buf.data_ptr(), G, qpk.D, qpk.precision, k1,
                  x["budget"], *x["own"], x["rank"].data_ptr(), x["S"].data_ptr(), x["sc"].data_ptr(), x["sc"].numel(), st)
    assert torch.equal(gather(lambda x: x["rank"]), ref["rank"])
    assert torch.equal(gather(lambda x: x["S"]).view(torch.int32), ref["S"].view(torch.int32))
    for x in ranks:
        _lib.call("ieee_gnn_stream_symbolic", x["rank"].data_ptr(), Q, G, k1, k2, *x["own"], x["sc"].data_ptr(), x["sc"].numel(), st)
    if k2 != 1:
        want_counts = counts_of(sc_ref, Q, G, k1, k2)
        for i in range(4):
            assert torch.equal(gather(lambda x: counts_of(x["sc"], Q, G, k1, k2)[i]), want_counts[i]), i
    for x in ranks:
        x["sizes"] = (C.c_int64 * 6)()
        _lib.call("ieee_gnn_stream_sizes_sync", Q, G, k1, k2, x["sc"].data_ptr(), x["sc"].numel(), x["sizes"], st)
        assert list(x["sizes"]) == list(sizes_ref)
        nnz, nnz_g, wb = x["sizes"][0], x["sizes"][1], x["sizes"][2]
        x.update(work=torch.empty(wb, dtype=torch.uint8, device=dev), a_ptr=torch.empty(N + 1, dtype=torch.int64, device=dev),
                 a_col=torch.empty(nnz, dtype=torch.int32, device=dev), a_val=torch.empty(nnz, dtype=torch.float32, device=dev),
                 g_ptr=torch.empty(N + 1, dtype=torch.int64, device=dev), g_row=torch.empty(nnz_g, dtype=torch.int32, device=dev),
                 g_val=torch.empty(nnz_g, dtype=torch.float32, device=dev))

    def numeric(step):
        for x in ranks:
            _lib.call("ieee_gnn_stream_numeric", step, x["rank"].data_ptr(), x["S"].data_ptr(), Q, G, k1, k2, *x["own"],
                      x["sc"].data_ptr(), x["sc"].numel(), x["work"].data_ptr(), x["work"].numel(), x["sizes"],
                      x["a_ptr"].data_ptr(), x["a_col"].data_ptr(), x["a_val"].data_ptr(), st)

    if k2 != 1:
        for step in range(3):
            numeric(step)
            for i in (2 * step, 2 * step + 1):
                summed(lambda x: work_arrays(x["work"], Q, G, k1, k2, x["sizes"])[i])
    numeric(3)
    lo = sizes_ref[0] - sizes_ref[1]
    for x in ranks:
        assert torch.equal(x["a_ptr"], ref["a_ptr"])
    summed(lambda x: x["a_col"][lo:])
    summed(lambda x: x["a_val"][lo:].view(torch.int32))
    for x in ranks:
        _lib.call("ieee_gnn_stream_csc", Q, G, k1, *x["own"], x["sc"].data_ptr(), x["sc"].numel(), x["a_ptr"].data_ptr(),
                  x["a_col"].data_ptr(), x["a_val"].data_ptr(), x["g_ptr"].data_ptr(), x["g_row"].data_ptr(),
                  x["g_val"].data_ptr(), st)
        assert torch.equal(x["g_ptr"], ref["g_ptr"])
    assert torch.equal(summed(lambda x: x["g_row"]), ref["g_row"])
    assert torch.equal(summed(lambda x: x["g_val"].view(torch.int32)), ref["g_val"].view(torch.int32))
    # A: each rank's own query rows, and the gallery rows everywhere
    a_col = ranks[0]["a_col"].clone()
    a_val = ranks[0]["a_val"].clone()
    for x in ranks:
        q0, q1 = x["own"][:2]
        p0, p1 = ref["a_ptr"][q0].item(), ref["a_ptr"][q1].item()
        a_col[p0:p1], a_val[p0:p1] = x["a_col"][p0:p1], x["a_val"][p0:p1]
    assert torch.equal(a_col, ref["a_col"]) and torch.equal(a_val.view(torch.int32), ref["a_val"].view(torch.int32))
    # each rank's query rows of the re-ranked distances, in blocks of 128
    for x in ranks:
        q0, q1 = x["own"][:2]
        out = torch.empty((q1 - q0, r32(G)), dtype=torch.float32, device=dev)
        acc = torch.empty(128 * G, dtype=torch.float64, device=dev)
        for s0 in range(q0, q1, 128):
            rows = min(128, q1 - s0)
            _lib.call("ieee_gnn_stream_block", x["a_ptr"].data_ptr(), x["a_col"].data_ptr(), x["a_val"].data_ptr(),
                      x["g_ptr"].data_ptr(), x["g_row"].data_ptr(), x["g_val"].data_ptr(), Q, G, s0, rows, out[s0 - q0].data_ptr(),
                      out.stride(0), acc.data_ptr(), 8 * acc.numel(), st)
        assert torch.equal(out[:, :G].view(torch.int32), want[q0:q1].contiguous().view(torch.int32)), x["own"]


CASES = {
    "26_7": dict(k1=26, k2=7),
    "10_1": dict(k1=10, k2=1),
    "12_12": dict(k1=12, k2=12),
    "bf16": dict(k1=26, k2=7, dtype=torch.bfloat16),
    "normalize_feature": dict(k1=26, k2=7, normalize=True),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("world", [2, 3, 8])
def test_phases_with_virtual_ranks(world, case):
    s = make_retrieval_set(300, 1700, 30, 4, dim=256, sigma=2.5, seed=world * 10 + len(case))     # Q not a multiple of 256
    run_virtual_ranks(s, world, **CASES[case])


@pytest.mark.parametrize("Q,G,k1,k2,world", [(5, 16, 21, 6, 2), (8, 13, 20, 20, 3), (6, 10, 15, 1, 2), (100, 1000, 26, 7, 3)])
def test_edge_shapes(Q, G, k1, k2, world):
    """k1 = N and k1 = N - 1; ranks that own no query rows, and (below 256 gallery rows) no gallery rows either."""
    s = make_retrieval_set(Q, G, 4, 2, dim=48, sigma=1.5, seed=Q * 100 + G)
    s.q_pids, s.g_pids = np.arange(Q, dtype=np.int64) % 2, np.arange(G, dtype=np.int64) % 2
    s.q_camids, s.g_camids = np.zeros(Q, dtype=np.int64), np.ones(G, dtype=np.int64)
    run_virtual_ranks(s, world, k1, k2)


def test_phase_argument_errors():
    lib = _lib.load()
    dev, st = torch.device("cuda"), _lib.stream()
    Q, G, k1, k2 = 300, 1700, 26, 7
    buf = torch.empty(1 << 22, dtype=torch.uint8, device=dev)
    p = buf.data_ptr()
    sizes = (C.c_int64 * 6)(1 << 20, 1 << 19, 0, 1 << 20, 1 << 20, 1 << 20)
    for own in ((0, 300, 100, 1700), (0, 200, 0, 1700), (0, 300, 0, 1800), (256, 0, 0, 1700), (0, 300, -256, 0)):
        calls = (lambda: lib.ieee_gnn_stream_neighbours_rows(p, Q, p, G, 64, 0, k1, 1 << 20, *own, p, p, p, buf.numel(), st),
                 lambda: lib.ieee_gnn_stream_symbolic(p, Q, G, k1, k2, *own, p, buf.numel(), st),
                 lambda: lib.ieee_gnn_stream_numeric(0, p, p, Q, G, k1, k2, *own, p, buf.numel(), p, buf.numel(), sizes, p, p, p, st),
                 lambda: lib.ieee_gnn_stream_csc(Q, G, k1, *own, p, buf.numel(), p, p, p, p, p, p, st))
        for call in calls:
            assert call() == _lib.ERR_INVALID and b"owned rows" in lib.ieee_last_error(), own
    own = (0, 300, 0, 1700)
    assert lib.ieee_gnn_stream_numeric(1, p, p, Q, G, k1, k2, *own, p, buf.numel(), p, 4096, sizes, p, p, p, st) == _lib.ERR_WORKSPACE
    assert lib.ieee_gnn_stream_csc(Q, G, k1, *own, p, 1024, p, p, p, p, p, p, st) == _lib.ERR_WORKSPACE
    assert lib.ieee_gnn_stream_symbolic(p, Q, G, k1, k2, *own, p, 1024, st) == _lib.ERR_WORKSPACE
    assert lib.ieee_gnn_stream_sizes_sync(Q, G, k1, k2, p, 1024, sizes, st) == _lib.ERR_WORKSPACE
    assert lib.ieee_gnn_stream_neighbours_rows(p, Q, p, G, 64, 0, k1, 1 << 20, *own, p, p, p, 1024, st) == _lib.ERR_WORKSPACE
    assert lib.ieee_gnn_stream_numeric(0, p, p, Q, G, k1, 1, *own, p, buf.numel(), p, buf.numel(), sizes, p, p, p, st) == \
        _lib.ERR_INVALID                                # k2 = 1 has step 3 only
    assert lib.ieee_gnn_stream_numeric(4, p, p, Q, G, k1, k2, *own, p, buf.numel(), p, buf.numel(), sizes, p, p, p, st) == \
        _lib.ERR_INVALID
    torch.cuda.synchronize()


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _init(rank, world, port):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    return dist


def _check_against_ungrouped(dist, s, k1=26, k2=7, block_bytes=None):
    """evaluate (twice: the second reuses the state and calls no phase) and ranked_lists of a query_group evaluator
    against an ungrouped one; the distance rows of every rank are all-gathered."""
    kw = {} if block_bytes is None else {"block_bytes": block_bytes}
    qf, gf = unit(s.qf).cuda(), unit(s.gf).cuda()
    Q, G = qf.shape[0], gf.shape[0]
    world, me = dist.get_world_size(), dist.get_rank()
    ref = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", k1=k1, k2=k2, **kw)
    c0, m0, i0 = ref.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    r0 = ref.ranked_lists(qf, s.q_pids, s.q_camids, k=15)
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", k1=k1, k2=k2, query_group=dist.group.WORLD, **kw)
    calls, real_call = [], _lib.call

    def spy(name, *args):
        calls.append(name)
        return real_call(name, *args)

    _lib.call = spy
    try:
        c1, m1, i1 = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        assert all(p in calls for p in PHASES) and "ieee_gnn_stream_graph" not in calls
        calls.clear()
        c2, m2, i2 = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        assert not any(p in calls for p in PHASES)                # the state is reused
        idx, val = ev.ranked_lists(qf, s.q_pids, s.q_camids, k=15)
        assert not any(p in calls for p in PHASES)
    finally:
        _lib.call = real_call
    owned = [rerank_owned(Q, G, world, r)[:2] for r in range(world)]
    for c, m, i in ((c1, m1, i1), (c2, m2, i2)):
        assert np.array_equal(c, c0) and m == m0 and i["mINP"] == i0["mINP"] and i["num_ties"] == i0["num_ties"]
        assert torch.equal(i["ap"], i0["ap"]) and torch.equal(i["first"], i0["first"])
        q0, q1 = owned[me]
        assert i["distmat"].shape == (q1 - q0, G)
        rows = max(b - a for a, b in owned)
        send = torch.zeros((rows, G), device="cuda")
        send[: q1 - q0] = i["distmat"]
        recv = torch.empty((world, rows, G), device="cuda")
        dist.all_gather_into_tensor(recv, send)
        d = torch.cat([recv[r, : b - a] for r, (a, b) in enumerate(owned)])
        assert torch.equal(d.view(torch.int32), i0["distmat"].view(torch.int32))
    assert torch.equal(idx, r0[0]) and torch.equal(val, r0[1])


def _errors(dist, s):
    gf = s.gf.cuda()
    grp = dist.group.WORLD
    with pytest.raises(ValueError, match="process group"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", query_group=object())
    with pytest.raises(ValueError, match="combined"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", query_group=grp, group=grp)
    for rerank in (False, True):
        with pytest.raises(ValueError, match="group="):
            RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank=rerank, query_group=grp)
    # the gallery-sharded route stays unsupported for GNN
    with pytest.raises(ValueError, match="sharded"):
        RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank="gnn", group=grp)


def _group_of_one_worker(rank, world, port, out):
    dist = _init(rank, world, port)
    s = make_retrieval_set(700, 2600, 50, 4, dim=192, sigma=2.5, seed=33)
    _check_against_ungrouped(dist, s, block_bytes=3 * 4 * 256 * 2600)       # 256-row query blocks: three of them
    _check_against_ungrouped(dist, make_retrieval_set(300, 1700, 30, 4, dim=128, sigma=2.5, seed=8), k1=10, k2=1)
    _errors(dist, s)
    # an empty query set behaves as without query_group
    outcomes = []
    for kw in ({}, {"query_group": dist.group.WORLD}):
        ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank="gnn", **kw)
        try:
            cmc, mAP, _ = ev.evaluate(s.qf[:0].cuda(), s.q_pids[:0], s.q_camids[:0])
            outcomes.append(("ok", cmc.tolist(), mAP))
        except Exception as e:            # noqa: BLE001 -- the ungrouped evaluator's own outcome is the reference
            outcomes.append((type(e).__name__, str(e)))
        idx, val = ev.ranked_lists(s.qf[:0].cuda(), k=5)
        assert idx.shape == (0, 5) and val.shape == (0, 5)
    assert outcomes[0] == outcomes[1]
    out[rank] = True
    dist.destroy_process_group()


def test_group_of_one():
    """A process group of one takes the shared code path (phases, exchanges, own query rows): the same bits as an
    evaluator without a group, and a second evaluation of the same queries runs no phase."""
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_group_of_one_worker, args=(1, _free_port(), out), nprocs=1, join=True)
    assert dict(out) == {0: True}


def _multi_gpu_worker(rank, world, port, out):
    dist = _init(rank, world, port)
    clustered = make_retrieval_set(700, 3001, 40, 4, dim=256, sigma=2.5, seed=17, distractor_frac=0.1)
    few = make_retrieval_set(200, 1500, 30, 4, dim=128, sigma=2.5, seed=5)           # Q <= 256: rank 1 evaluates nothing
    _check_against_ungrouped(dist, clustered, block_bytes=3 * 4 * 256 * 3001)
    _check_against_ungrouped(dist, few)
    _check_against_ungrouped(dist, few, k1=10, k2=1)
    _errors(dist, few)
    gf = few.gf.cuda()
    # settings that differ between the ranks: every rank raises, none waits for the others
    with pytest.raises(ValueError, match="disagree"):
        RetrievalEvaluator(gf, few.g_pids, few.g_camids, rerank="gnn", k1=26 + rank, query_group=dist.group.WORLD)
    with pytest.raises(ValueError, match="disagree"):
        RetrievalEvaluator(gf[: 1500 - rank], few.g_pids[: 1500 - rank], few.g_camids[: 1500 - rank], rerank="gnn",
                           query_group=dist.group.WORLD)
    ev = RetrievalEvaluator(gf, few.g_pids, few.g_camids, rerank="gnn", query_group=dist.group.WORLD,
                            block_bytes=(1 << 26) * (1 + rank))          # block_bytes may differ
    Q = 200 - rank
    with pytest.raises(ValueError, match="different numbers of queries"):
        ev.evaluate(unit(few.qf[:Q]).cuda(), few.q_pids[:Q], few.q_camids[:Q])
    dist.barrier()
    out[rank] = True
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_query_group():
    """GNN re-ranking shared by two GPUs, on a set with several query blocks per rank and on one where rank 1 owns no
    query: the all-gathered distance rows, cmc, mAP, mINP, ap, first and ranked lists equal one GPU's."""
    import torch.multiprocessing as mp
    world = 2
    out = mp.Manager().dict()
    mp.spawn(_multi_gpu_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert dict(out) == {r: True for r in range(world)}
