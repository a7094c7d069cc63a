"""k-reciprocal re-ranking over a sharded gallery (RetrievalEvaluator(group=..., rerank=True)): the library's phases
with virtual ranks on one GPU, the Python plumbing in a process group of one, and -- when the box has two GPUs -- the
real thing over NCCL with both exchanges, all bit for bit against one GPU holding the whole gallery."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

from ieee_b200 import _lib
from ieee_b200.engine import PackedFeatures, RetrievalEvaluator, packed_distmat, rerank_owned, shard_bounds
from ieee_b200.testing import make_retrieval_set, rgbnt201_shaped

pytestmark = pytest.mark.gpu


def strip_budget(Q, G, k1, width):
    r32 = lambda x: (x + 31) // 32 * 32
    return width * 4 * (Q + r32(G) + r32(Q + G) + k1 + 1)


def v_arrays(ws, Q, G, k1, k2):
    """(columns, values as int32 bits, counts) of V in a workspace, valid entries only."""
    cap, oc, ov, on = C.c_int64(), C.c_size_t(), C.c_size_t(), C.c_size_t()
    _lib.call("ieee_rerank_stream_v_layout", Q, G, k1, k2, C.byref(cap), C.byref(oc), C.byref(ov), C.byref(on))
    N, c = Q + G, cap.value
    col = ws[oc.value: oc.value + 4 * N * c].view(torch.int32).view(N, c)
    val = ws[ov.value: ov.value + 4 * N * c].view(torch.int32).view(N, c)
    cnt = ws[on.value: on.value + 4 * N].view(torch.int32)
    mask = torch.arange(c, device=ws.device)[None, :] < cnt[:, None]
    return col[mask], val[mask], cnt.clone(), val.view(torch.float32)


CASES = {
    "euclidean": dict(k1=20, k2=6, lam=0.3),
    "k2_is_1": dict(k1=20, k2=1, lam=0.0),
    "cosine_normalized_lambda_1": dict(k1=12, k2=4, lam=1.0, metric="cosine", normalize=True),
    "bf16": dict(k1=20, k2=6, lam=0.3, dtype=torch.bfloat16),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("shards", [2, 3, 8])
def test_phases_with_virtual_ranks(shards, case):
    """Each virtual rank runs the passes on its own samples (at its own strip width), the owned rows are merged as the
    all-gathers would merge them, and each rank finishes and blends its own gallery window (shard_bounds: not aligned
    to 128).  colmax, rank, V and every window's re-ranked columns equal the one-GPU prepare and block calls."""
    kw = CASES[case]
    k1, k2, lam = kw["k1"], kw["k2"], kw["lam"]
    Q, G = 300, 1700                                     # Q is not a multiple of 256
    s = make_retrieval_set(Q, G, 30, 4, dim=192, sigma=2.5, seed=shards * 10 + len(case))
    dtype = kw.get("dtype", torch.float32)
    qf, gf = s.qf.cuda().to(dtype), s.gf.cuda().to(dtype)
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, kw.get("metric", "euclidean"), kw.get("normalize", False), rerank=True,
                            k1=k1, k2=k2, lambda_value=lam)
    ev.evaluate(qf, s.q_pids, s.q_camids)                # fixes the centre and prepares the one-GPU state
    ref = ev._rr
    qpk = PackedFeatures(qf, ev.metric, ev.normalize, ev.precision, ev.center)
    gpk = PackedFeatures(gf, ev.metric, ev.normalize, ev.precision, ev.center)
    dev, N, lib = qf.device, Q + G, _lib.load()
    qg = packed_distmat(qpk, gpk, torch.empty((Q, G), dtype=torch.float32, device=dev))
    want = qg.clone()
    acc = torch.empty(Q * G, dtype=torch.float32, device=dev)
    _lib.call("ieee_rerank_stream_block", ref["ws"].data_ptr(), Q, G, k1, k2, ref["colmax"].data_ptr(), 0, Q, lam,
              want.data_ptr(), want.stride(0), acc.data_ptr(), 4 * acc.numel(), _lib.stream())

    ranks = []
    for r in range(shards):
        g_lo, g_hi = shard_bounds(G, shards, r)
        ws_bytes = lib.ieee_rerank_stream_window_workspace_bytes(Q, G, k1, k2, g_hi - g_lo)
        budget = strip_budget(Q, G, k1, 256 * (1 + r % 3))
        sc_bytes = lib.ieee_rerank_stream_scratch_bytes(Q, G, k1, budget)
        ranks.append(dict(window=(g_lo, g_hi), own=rerank_owned(Q, G, shards, r), budget=budget,
                          ws=torch.empty(ws_bytes, dtype=torch.uint8, device=dev),
                          sc=torch.empty(sc_bytes, dtype=torch.uint8, device=dev),
                          colmax=torch.full((N,), float("nan"), device=dev),
                          rank=torch.full((N, k1 + 1), -7, dtype=torch.int32, device=dev)))

    def run_pass(step):
        for x in ranks:
            q0, q1, g0, g1 = x["own"]
            _lib.call("ieee_rerank_stream_pass", step, qpk.buf.data_ptr(), Q, gpk.buf.data_ptr(), G, qpk.D, qpk.metric,
                      qpk.precision, k1, k2, x["budget"], q0, q1, g0, g1, x["colmax"].data_ptr(), x["rank"].data_ptr(),
                      x["ws"].data_ptr(), x["ws"].numel(), x["sc"].data_ptr(), x["sc"].numel(), _lib.stream())

    def merge(get):
        """What the all-gather of the owned rows leaves on every rank."""
        full = get(ranks[0]).clone()
        for x in ranks:
            q0, q1, g0, g1 = x["own"]
            full[q0:q1] = get(x)[q0:q1]
            full[Q + g0: Q + g1] = get(x)[Q + g0: Q + g1]
        for x in ranks:
            get(x).copy_(full)
        return full

    run_pass(0)
    colmax, rank = merge(lambda x: x["colmax"]), merge(lambda x: x["rank"])
    assert torch.equal(colmax.view(torch.int32), ref["colmax"].view(torch.int32))
    assert torch.equal(rank, ref["rank"])
    run_pass(1)
    merged = merge(lambda x: v_arrays(x["ws"], Q, G, k1, k2)[3])
    col_r, val_r, cnt_r, _ = v_arrays(ref["ws"], Q, G, k1, k2)
    for x in ranks:                                      # membership: every rank computes all rows itself
        col, val, cnt, _ = v_arrays(x["ws"], Q, G, k1, k2)
        assert torch.equal(cnt, cnt_r) and torch.equal(col, col_r) and torch.equal(val, val_r)
    assert merged.shape[0] == N
    for x in ranks:
        g_lo, g_hi = x["window"]
        Gs = g_hi - g_lo
        _lib.call("ieee_rerank_stream_finish", x["ws"].data_ptr(), x["ws"].numel(), Q, G, k1, k2, g_lo, Gs, x["rank"].data_ptr(),
                  _lib.stream())
        blk = qg[:, g_lo:g_hi].contiguous()
        scratch = torch.empty(128 * Gs, dtype=torch.float32, device=dev)
        for row0 in range(0, Q, 128):                    # several query blocks
            rows = min(128, Q - row0)
            _lib.call("ieee_rerank_stream_block_window", x["ws"].data_ptr(), Q, G, k1, k2, Gs, x["colmax"].data_ptr(), row0,
                      rows, lam, blk[row0].data_ptr(), blk.stride(0), scratch.data_ptr(), 4 * scratch.numel(), _lib.stream())
        assert torch.equal(blk.view(torch.int32), want[:, g_lo:g_hi].contiguous().view(torch.int32)), x["window"]


def test_phase_argument_errors():
    lib = _lib.load()
    dev = torch.device("cuda")
    Q, G, k1, k2 = 300, 1700, 20, 6
    buf = torch.empty(1 << 20, dtype=torch.uint8, device=dev)
    for own in ((0, 300, 100, 1700), (0, 200, 0, 1700), (0, 300, 0, 1800), (256, 0, 0, 1700)):
        rc = lib.ieee_rerank_stream_pass(0, buf.data_ptr(), Q, buf.data_ptr(), G, 64, 0, 0, k1, k2, 1 << 20, *own,
                                         buf.data_ptr(), buf.data_ptr(), None, 0, buf.data_ptr(), buf.numel(), _lib.stream())
        assert rc == _lib.ERR_INVALID and b"owned samples" in lib.ieee_last_error(), own
    rc = lib.ieee_rerank_stream_finish(buf.data_ptr(), buf.numel(), Q, G, k1, k2, 1000, 701, buf.data_ptr(), _lib.stream())
    assert rc == _lib.ERR_INVALID and b"window" in lib.ieee_last_error()
    rc = lib.ieee_rerank_stream_finish(buf.data_ptr(), 1024, Q, G, k1, k2, 0, G, buf.data_ptr(), _lib.stream())
    assert rc == _lib.ERR_WORKSPACE


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


def _group_of_one_worker(rank, world, port, out):
    dist = _init(rank, world, port)
    s = make_retrieval_set(700, 2600, 50, 4, dim=192, sigma=2.5, seed=33)
    G = 2600
    qf = s.qf.cuda()
    block_bytes = 2 * 4 * 256 * G                        # 256-row query blocks: three of them
    ref = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True, block_bytes=block_bytes)
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True, block_bytes=block_bytes, group=dist.group.WORLD,
                            g_offset=0, g_total=G)
    c0, m0, i0 = ref.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    calls, real_call = [], _lib.call

    def spy(name, *args):
        calls.append(name)
        return real_call(name, *args)

    _lib.call = spy
    try:
        c1, m1, i1 = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        assert "ieee_rerank_stream_pass" in calls and "ieee_rerank_stream_prepare" not in calls
        calls.clear()
        c2, m2, i2 = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        assert "ieee_rerank_stream_pass" not in calls and "ieee_rerank_stream_finish" not in calls    # the state is reused
    finally:
        _lib.call = real_call
    for c, m, i in ((c1, m1, i1), (c2, m2, i2)):
        assert np.array_equal(c, c0) and m == m0 and i["mINP"] == i0["mINP"]
        assert torch.equal(i["distmat"], i0["distmat"]) and torch.equal(i["ap"], i0["ap"]) and torch.equal(i["first"], i0["first"])
    a, b = ev.ranked_lists(qf, s.q_pids, s.q_camids, k=15), ref.ranked_lists(qf, s.q_pids, s.q_camids, k=15)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    with pytest.raises(ValueError, match="tile"):
        RetrievalEvaluator(s.gf[3:].cuda(), s.g_pids[3:], s.g_camids[3:], rerank=True, group=dist.group.WORLD, g_offset=3,
                           g_total=G)
    with pytest.raises(ValueError, match="sharded"):
        RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank="gnn", group=dist.group.WORLD)
    out[rank] = True
    dist.destroy_process_group()


def test_group_of_one():
    """A process group of one takes the sharded code path (gather, phases, exchanges, windowed blocks): the same bits as
    an evaluator without a group, and a second evaluation of the same queries does not prepare again."""
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_group_of_one_worker, args=(1, _free_port(), out), nprocs=1, join=True)
    assert dict(out) == {0: True}


def _data_sets(world):
    """(name, set, slice bounds of every rank): q == g with slices starting at multiples of 128, and a clustered set with
    the default shard_bounds split."""
    c3 = rgbnt201_shaped()
    G = c3.gf.shape[0]
    cuts = [0] + [(G * r // world) // 128 * 128 for r in range(1, world)] + [G]
    clustered = make_retrieval_set(500, 3001, 40, 4, dim=256, sigma=2.5, seed=17, distractor_frac=0.1)
    return [("rgbnt201", c3, [(cuts[r], cuts[r + 1]) for r in range(world)]),
            ("clustered", clustered, [shard_bounds(3001, world, r) for r in range(world)])]


def _multi_gpu_worker(rank, world, port, out):
    dist = _init(rank, world, port)
    for name, s, bounds in _data_sets(world):
        G = s.gf.shape[0]
        qf = s.qf.cuda()
        g0, g1 = bounds[rank]
        block_bytes = 2 * 4 * 256 * max(b - a for a, b in bounds)        # the same 256-row query blocks on every rank
        ref = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True)
        c0, m0, i0 = ref.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        r0 = ref.ranked_lists(qf, s.q_pids, s.q_camids, k=20)
        for exchange in ("peer", "nccl"):
            ev = RetrievalEvaluator(s.gf[g0:g1].cuda(), s.g_pids[g0:g1], s.g_camids[g0:g1], rerank=True, group=dist.group.WORLD,
                                    g_offset=g0, g_total=G, block_bytes=block_bytes, exchange=exchange)
            c, m, i = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
            parts = [torch.empty((qf.shape[0], b - a), device="cuda") for a, b in bounds]
            dist.all_gather(parts, i["distmat"].contiguous())
            d = torch.cat(parts, 1)
            assert torch.equal(d.view(torch.int32), i0["distmat"].view(torch.int32)), (name, exchange)
            assert np.array_equal(c, c0) and m == m0 and i["mINP"] == i0["mINP"], (name, exchange)
            assert torch.equal(i["ap"], i0["ap"]) and torch.equal(i["first"], i0["first"]), (name, exchange)
            idx, val = ev.ranked_lists(qf, s.q_pids, s.q_camids, k=20)
            assert torch.equal(idx, r0[0]) and torch.equal(val, r0[1]), (name, exchange)
    # slices with a gap: every rank raises, none waits for the others
    s = _data_sets(world)[1][1]
    g0, g1 = shard_bounds(3001, world, rank)
    lo = g0 + (1 if rank == world - 1 else 0)
    with pytest.raises(ValueError, match="tile"):
        RetrievalEvaluator(s.gf[lo:g1].cuda(), s.g_pids[lo:g1], s.g_camids[lo:g1], rerank=True, group=dist.group.WORLD,
                           g_offset=lo, g_total=3001)
    dist.barrier()
    out[rank] = True
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_sharded_rerank():
    """Re-ranking over a gallery sharded across two GPUs, with the peer and the NCCL exchange and several query blocks:
    the all-gathered distances, cmc, mAP, mINP, ap, first and ranked lists equal one GPU's."""
    import torch.multiprocessing as mp
    world = 2
    out = mp.Manager().dict()
    mp.spawn(_multi_gpu_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert dict(out) == {r: True for r in range(world)}
