"""k-reciprocal re-ranking over a sharded gallery with every strip computed by all ranks together, none holding the
whole gallery (ieee_rerank_stream_part_*): the library's calls with virtual ranks on one GPU and the collectives done in
Python, the evaluator's prepare in a process group of one (with a spy on the collectives) and in a gloo group of three
processes sharing one GPU, and -- when the box has two GPUs -- the whole evaluation over NCCL.  All bit for bit against
one GPU holding the whole gallery."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

from ieee_b200 import _lib
from ieee_b200.engine import PackedFeatures, RetrievalEvaluator, packed_distmat, rerank_owned, rerank_ranges, shard_bounds
from ieee_b200.testing import make_retrieval_set

pytestmark = pytest.mark.gpu

CASES = {
    "euclidean": dict(k1=20, k2=6, lam=0.3),
    "k2_is_1": dict(k1=20, k2=1, lam=0.0),
    "cosine_normalized_lambda_1": dict(k1=12, k2=4, lam=1.0, metric="cosine", normalize=True),
    "bf16": dict(k1=20, k2=6, lam=0.3, dtype=torch.bfloat16),
}


def v_arrays(ws, Q, G, k1, k2):
    """(columns, values as int32 bits, counts) of V in a workspace, valid entries only, and the [N, cap] value rows."""
    cap, oc, ov, on = C.c_int64(), C.c_size_t(), C.c_size_t(), C.c_size_t()
    _lib.call("ieee_rerank_stream_v_layout", Q, G, k1, k2, C.byref(cap), C.byref(oc), C.byref(ov), C.byref(on))
    N, c = Q + G, cap.value
    col = ws[oc.value: oc.value + 4 * N * c].view(torch.int32).view(N, c)
    val = ws[ov.value: ov.value + 4 * N * c].view(torch.int32).view(N, c)
    cnt = ws[on.value: on.value + 4 * N].view(torch.int32)
    mask = torch.arange(c, device=ws.device)[None, :] < cnt[:, None]
    return col[mask], val[mask], cnt.clone(), val


def slice_sizes(layout, G, shards):
    if layout == "shard_bounds":
        return [b - a for a, b in (shard_bounds(G, shards, r) for r in range(shards))]
    return [30] * (shards - 1) + [G - 30 * (shards - 1)]      # "short": every range but the first and the last empty


def strips(Q, G, W):
    for i0, n in ((0, Q), (Q, G)):
        for c0 in range(0, n, W):
            yield i0 + c0, min(W, n - c0)


@pytest.mark.parametrize("layout", ["shard_bounds", "short"])
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("shards", [1, 2, 3, 8])
def test_part_calls_with_virtual_ranks(shards, case, layout):
    """Each virtual rank contracts its part of every strip (its queries of rerank_owned, its gallery range of
    rerank_ranges); the collectives are done here as the evaluator does them (MAX of colmax bits, all-gather + merge of
    the lists, int32 sum of V's value rows).  colmax, rank, V and every slice's re-ranked columns equal the one-GPU
    prepare and block calls."""
    kw = CASES[case]
    k1, k2, lam = kw["k1"], kw["k2"], kw["lam"]
    Q, G = 300, 1700
    if layout == "short" and shards == 1:
        pytest.skip("one rank holds the whole gallery")
    s = make_retrieval_set(Q, G, 30, 4, dim=192, sigma=2.5, seed=shards * 10 + len(case))
    dtype = kw.get("dtype", torch.float32)
    qf, gf = s.qf.cuda().to(dtype), s.gf.cuda().to(dtype)
    ev = RetrievalEvaluator(gf, s.g_pids, s.g_camids, kw.get("metric", "euclidean"), kw.get("normalize", False), rerank=True,
                            k1=k1, k2=k2, lambda_value=lam)
    ev.evaluate(qf, s.q_pids, s.q_camids)                # fixes the centre and prepares the one-GPU state
    ref = ev._rr
    pack = lambda t: PackedFeatures(t, ev.metric, ev.normalize, ev.precision, ev.center)
    qpk, gpk = pack(qf), pack(gf)
    dev, N, k1p, lib, stream = qf.device, Q + G, k1 + 1, _lib.load(), _lib.stream()
    qg = packed_distmat(qpk, gpk, torch.empty((Q, G), dtype=torch.float32, device=dev))
    want = qg.clone()
    acc = torch.empty(Q * G, dtype=torch.float32, device=dev)
    _lib.call("ieee_rerank_stream_block", ref["ws"].data_ptr(), Q, G, k1, k2, ref["colmax"].data_ptr(), 0, Q, lam,
              want.data_ptr(), want.stride(0), acc.data_ptr(), 4 * acc.numel(), _lib.stream())

    sizes = slice_sizes(layout, G, shards)
    offsets = [sum(sizes[:r]) for r in range(shards)]
    ranges = rerank_ranges(offsets, G)
    parts = [rerank_owned(Q, G, shards, r)[:2] + ranges[r] for r in range(shards)]
    budgets = [(1 + r % 3) << 20 for r in range(shards)]           # the ranks' own budgets differ; they share the narrowest
    W = min(lib.ieee_rerank_stream_part_width(Q, G, k1, *p, b) for p, b in zip(parts, budgets))
    assert W >= 256 and W % 256 == 0
    ranks = []
    for r, p in enumerate(parts):
        sc_bytes = lib.ieee_rerank_stream_part_scratch_bytes(Q, G, k1, *p, W)
        ws_bytes = lib.ieee_rerank_stream_window_workspace_bytes(Q, G, k1, k2, sizes[r])
        ranks.append(dict(part=p, window=(offsets[r], sizes[r]), gpart=pack(gf[p[2]:p[3]]) if p[3] > p[2] else None,
                          sc=torch.empty(sc_bytes, dtype=torch.uint8, device=dev),
                          ws=torch.empty(ws_bytes, dtype=torch.uint8, device=dev),
                          colmax=torch.full((N,), float("nan"), device=dev),
                          rank=torch.full((N, k1p), -7, dtype=torch.int32, device=dev)))

    def contract(step, x, i0, wc, g_strip):
        _lib.call("ieee_rerank_stream_part_contract", step, qpk.buf.data_ptr(), Q, _lib.ptr(x["gpart"] and x["gpart"].buf),
                  _lib.ptr(g_strip and g_strip.buf), G, qpk.D, qpk.metric, qpk.precision, k1, *x["part"], W, i0, wc,
                  x["colmax"].data_ptr(), x["sc"].data_ptr(), x["sc"].numel(), stream)

    for i0, wc in strips(Q, G, W):                       # pass 0
        g_strip = pack(gf[i0 - Q: i0 - Q + wc]) if i0 >= Q else None
        for x in ranks:
            contract(0, x, i0, wc, g_strip)
        cm = torch.stack([x["colmax"][i0:i0 + wc].view(torch.int32) for x in ranks]).amax(0)
        idx, val = [], []
        for x in ranks:
            x["colmax"][i0:i0 + wc] = cm.view(torch.float32)
            li = torch.empty(2 * wc * k1p, dtype=torch.int32, device=dev)
            lv = torch.empty(2 * wc * k1p, dtype=torch.float32, device=dev)
            _lib.call("ieee_rerank_stream_part_topk", Q, G, k1, *x["part"], W, i0, wc, x["colmax"].data_ptr(), li.data_ptr(),
                      lv.data_ptr(), x["sc"].data_ptr(), x["sc"].numel(), stream)
            idx.append(li)
            val.append(lv)
        idx, val = torch.cat(idx), torch.cat(val)
        merged_val = torch.empty(wc * k1p, dtype=torch.float32, device=dev)
        for x in ranks:
            _lib.call("ieee_topk_merge", idx.data_ptr(), val.data_ptr(), 2 * shards, wc, k1p, x["rank"][i0].data_ptr(),
                      merged_val.data_ptr(), stream)
    for x in ranks:
        assert torch.equal(x["colmax"].view(torch.int32), ref["colmax"].view(torch.int32))
        assert torch.equal(x["rank"], ref["rank"])

    for x in ranks:                                      # pass 1: membership of every row, no strips
        _lib.call("ieee_rerank_stream_pass", 1, qpk.buf.data_ptr(), Q, None, G, qpk.D, qpk.metric, qpk.precision, k1, k2, 0,
                  0, 0, 0, 0, x["colmax"].data_ptr(), x["rank"].data_ptr(), x["ws"].data_ptr(), x["ws"].numel(), None, 0, stream)
    for i0, wc in strips(Q, G, W):
        g_strip = pack(gf[i0 - Q: i0 - Q + wc]) if i0 >= Q else None
        for x in ranks:
            contract(1, x, i0, wc, g_strip)
            _lib.call("ieee_rerank_stream_part_members", Q, G, k1, k2, *x["part"], W, i0, wc, x["colmax"].data_ptr(),
                      x["ws"].data_ptr(), x["ws"].numel(), x["sc"].data_ptr(), x["sc"].numel(), stream)
        rows = [v_arrays(x["ws"], Q, G, k1, k2)[3][i0:i0 + wc] for x in ranks]
        nonzero = torch.stack([(r != 0).to(torch.int32) for r in rows]).sum(0)
        assert int(nonzero.max()) <= 1                   # one contributor per entry: the int32 sum is exact
        total = torch.stack(rows).to(torch.int64).sum(0).to(torch.int32)
        for x, r in zip(ranks, rows):
            r.copy_(total)
            _lib.call("ieee_rerank_stream_part_weights", x["ws"].data_ptr(), x["ws"].numel(), Q, G, k1, k2, i0, wc, stream)
    col_r, val_r, cnt_r, _ = v_arrays(ref["ws"], Q, G, k1, k2)
    for x in ranks:
        col, val, cnt, _ = v_arrays(x["ws"], Q, G, k1, k2)
        assert torch.equal(cnt, cnt_r) and torch.equal(col, col_r) and torch.equal(val, val_r)

    for x in ranks:                                      # finish and blend each rank's slice
        g_lo, Gs = x["window"]
        _lib.call("ieee_rerank_stream_finish", x["ws"].data_ptr(), x["ws"].numel(), Q, G, k1, k2, g_lo, Gs, x["rank"].data_ptr(),
                  stream)
        if Gs == 0:
            continue
        blk = qg[:, g_lo:g_lo + Gs].contiguous()
        scratch = torch.empty(128 * Gs, dtype=torch.float32, device=dev)
        for row0 in range(0, Q, 128):
            n = min(128, Q - row0)
            _lib.call("ieee_rerank_stream_block_window", x["ws"].data_ptr(), Q, G, k1, k2, Gs, x["colmax"].data_ptr(), row0, n,
                      lam, blk[row0].data_ptr(), blk.stride(0), scratch.data_ptr(), 4 * scratch.numel(), stream)
        assert torch.equal(blk.view(torch.int32), want[:, g_lo:g_lo + Gs].contiguous().view(torch.int32)), x["window"]


def test_part_argument_errors():
    lib = _lib.load()
    dev = torch.device("cuda")
    Q, G, k1, k2 = 300, 1700, 20, 6
    buf = torch.empty(1 << 24, dtype=torch.uint8, device=dev)
    p, st = buf.data_ptr(), _lib.stream()
    good = (0, 300, 0, 1700)

    def contract(part=good, W=256, i0=0, wc=256, nbytes=buf.numel(), step=0):
        return lib.ieee_rerank_stream_part_contract(step, p, Q, p, p, G, 64, 0, 0, k1, *part, W, i0, wc, p, p, nbytes, st)

    for part in ((0, 301, 0, 1700), (0, 300, 100, 1700), (0, 300, 0, 1701), (200, 100, 0, 1700)):
        assert contract(part=part) == _lib.ERR_INVALID, part
        assert b"part" in lib.ieee_last_error()
    assert contract(W=300) == _lib.ERR_INVALID and b"strip width" in lib.ieee_last_error()
    for i0, wc in ((100, 100), (Q + 100, 100), (0, 512), (256, 256), (Q + 1536, 256)):
        assert contract(i0=i0, wc=wc) == _lib.ERR_INVALID and b"strip" in lib.ieee_last_error(), (i0, wc)
    assert contract(step=2) == _lib.ERR_INVALID and b"pass" in lib.ieee_last_error()
    assert contract(nbytes=1024) == _lib.ERR_WORKSPACE and b"too small" in lib.ieee_last_error()
    rc = lib.ieee_rerank_stream_part_topk(Q, G, k1, 0, 300, 128, 1700, 256, 0, 256, p, p, p, p, buf.numel(), st)
    assert rc == _lib.ERR_INVALID and b"multiple of 256" in lib.ieee_last_error()
    rc = lib.ieee_rerank_stream_part_topk(Q, G, k1, *good, 256, 0, 256, p, p, p, p, 1024, st)
    assert rc == _lib.ERR_WORKSPACE
    rc = lib.ieee_rerank_stream_part_members(Q, G, k1, k2, *good, 512, 0, 300, p, p, 1024, p, buf.numel(), st)
    assert rc == _lib.ERR_WORKSPACE and b"workspace too small" in lib.ieee_last_error()
    rc = lib.ieee_rerank_stream_part_members(Q, G, k1, k2, *good, 512, 0, 300, p, p, buf.numel(), p, 1024, st)
    assert rc == _lib.ERR_WORKSPACE and b"scratch too small" in lib.ieee_last_error()
    rc = lib.ieee_rerank_stream_part_weights(p, buf.numel(), Q, G, k1, k2, 1900, 200, st)
    assert rc == _lib.ERR_INVALID and b"rows" in lib.ieee_last_error()
    rc = lib.ieee_rerank_stream_part_weights(p, 1024, Q, G, k1, k2, 0, 200, st)
    assert rc == _lib.ERR_WORKSPACE


def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _init(backend, rank, world, port, device):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(device)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", device))
    else:
        dist.init_process_group(backend, rank=rank, world_size=world)
    return dist


def _group_of_one_worker(rank, world, port, out):
    dist = _init("nccl", rank, world, port, rank)
    s = make_retrieval_set(700, 2600, 50, 4, dim=192, sigma=2.5, seed=34)
    G, D, k1 = 2600, 192, 20
    qf = s.qf.cuda()
    block_bytes = 2 * 4 * 256 * G
    ref = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True, block_bytes=block_bytes)
    ev = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True, block_bytes=block_bytes, group=dist.group.WORLD,
                            g_offset=0, g_total=G)
    c0, m0, i0 = ref.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    ev.evaluate(qf.clone(), s.q_pids, s.q_camids)       # fixes the centre and packs the slice
    W = _lib.load().ieee_rerank_stream_part_width(qf.shape[0], G, k1, 0, qf.shape[0], 0, G, block_bytes)
    assert W < G
    moved, real = [], {}

    def spy(name):
        fn = real[name] = getattr(dist, name)

        def wrapped(*args, **kwargs):
            moved.append((name, max(a.numel() * a.element_size() for a in args if isinstance(a, torch.Tensor))))
            return fn(*args, **kwargs)
        setattr(dist, name, wrapped)

    for name in ("all_reduce", "all_gather_into_tensor", "all_gather", "broadcast", "reduce_scatter_tensor"):
        spy(name)
    try:
        ev._rerank_prepare(qf)
    finally:
        for name, fn in real.items():
            setattr(dist, name, fn)
    torch.cuda.synchronize()
    cap, oc, ov, on = C.c_int64(), C.c_size_t(), C.c_size_t(), C.c_size_t()
    _lib.call("ieee_rerank_stream_v_layout", qf.shape[0], G, k1, 6, C.byref(cap), C.byref(oc), C.byref(ov), C.byref(on))
    strip_bytes, list_bytes, v_bytes = W * D * 4, 2 * W * (k1 + 1) * 4, W * cap.value * 4
    assert moved and max(n for _, n in moved) <= max(strip_bytes, list_bytes, v_bytes), moved
    assert max(n for _, n in moved) < G * D * 4                # far from the whole gallery
    c1, m1, i1 = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)   # the state prepared above
    assert np.array_equal(c1, c0) and m1 == m0 and i1["mINP"] == i0["mINP"]
    for k in ("distmat", "ap", "first"):
        assert torch.equal(i1[k], i0[k]), k
    a, b = ev.ranked_lists(qf, s.q_pids, s.q_camids, k=15), ref.ranked_lists(qf, s.q_pids, s.q_camids, k=15)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    out[rank] = True
    dist.destroy_process_group()


def test_group_of_one_moves_one_strip_at_a_time():
    """In a process group of one the prepare's collectives carry at most one gallery strip's rows or one strip's
    neighbour lists, never the gallery, and the results equal an evaluator without a group bit for bit."""
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_group_of_one_worker, args=(1, _free_port(), out), nprocs=1, join=True)
    assert dict(out) == {0: True}


SIZES_3 = [100, 800, 800]          # ranges [0, 256), [256, 1024), [1024, 1700): two of them reach into the next slice


def _gloo_worker(rank, world, port, out):
    dist = _init("gloo", rank, world, port, 0)
    Q, G, k1, k2, lam = 300, 1700, 20, 6, 0.3
    s = make_retrieval_set(Q, G, 30, 4, dim=192, sigma=2.5, seed=71)
    qf, gf = s.qf.cuda(), s.gf.cuda()
    ref = RetrievalEvaluator(gf, s.g_pids, s.g_camids, rerank=True, k1=k1, k2=k2, lambda_value=lam)
    ref.evaluate(qf, s.q_pids, s.q_camids)
    off = sum(SIZES_3[:rank])
    n = SIZES_3[rank]
    budget = (1 + rank) * 2 ** 20
    ev = RetrievalEvaluator(gf[off:off + n], s.g_pids[off:off + n], s.g_camids[off:off + n], rerank=True, k1=k1, k2=k2,
                            lambda_value=lam, group=dist.group.WORLD, g_offset=off, g_total=G, center=ref.center,
                            block_bytes=budget)
    rr = ev._rerank_prepare(qf)
    torch.cuda.synchronize()
    assert torch.equal(rr["colmax"].view(torch.int32), ref._rr["colmax"].view(torch.int32))
    assert torch.equal(rr["rank"], ref._rr["rank"])
    mine, theirs = v_arrays(rr["ws"], Q, G, k1, k2), v_arrays(ref._rr["ws"], Q, G, k1, k2)
    assert all(torch.equal(a, b) for a, b in zip(mine[:3], theirs[:3]))
    qpk = PackedFeatures(qf, ref.metric, ref.normalize, ref.precision, ref.center)
    gpk = PackedFeatures(gf, ref.metric, ref.normalize, ref.precision, ref.center)
    qg = packed_distmat(qpk, gpk, torch.empty((Q, G), dtype=torch.float32, device=qf.device))
    want = ref._rerank_block(qg.clone(), 0)
    got = ev._rerank_block(qg[:, off:off + n].contiguous(), 0)
    assert torch.equal(got.view(torch.int32), want[:, off:off + n].contiguous().view(torch.int32))
    out[rank] = True
    dist.barrier()
    dist.destroy_process_group()


def test_three_ranks_sharing_one_gpu():
    """Three processes of a gloo group on one GPU, with slices whose aligned ranges need rows of the next slices and with
    different block_bytes: every rank's prepared state (colmax, rank, V) and its slice's re-ranked distances equal one
    GPU's."""
    import torch.multiprocessing as mp
    world = len(SIZES_3)
    out = mp.Manager().dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert dict(out) == {r: True for r in range(world)}


def _multi_gpu_worker(rank, world, port, out):
    dist = _init("nccl", rank, world, port, rank)
    s = make_retrieval_set(500, 3001, 40, 4, dim=2048, sigma=2.5, seed=19, distractor_frac=0.1)
    G = 3001
    bounds = [shard_bounds(G, world, r) for r in range(world)]
    qf = s.qf.cuda()
    g0, g1 = bounds[rank]
    block_bytes = 2 * 4 * 256 * max(b - a for a, b in bounds)
    ref = RetrievalEvaluator(s.gf.cuda(), s.g_pids, s.g_camids, rerank=True)
    c0, m0, i0 = ref.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
    r0 = ref.ranked_lists(qf, s.q_pids, s.q_camids, k=20)
    whole_packed = PackedFeatures(s.gf.cuda(), ref.metric, ref.normalize, ref.precision, ref.center).buf.numel()
    for exchange in ("peer", "nccl"):
        ev = RetrievalEvaluator(s.gf[g0:g1].cuda(), s.g_pids[g0:g1], s.g_camids[g0:g1], rerank=True, group=dist.group.WORLD,
                                g_offset=g0, g_total=G, block_bytes=block_bytes, exchange=exchange, center=ref.center)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        rr = ev._rerank_prepare(qf)
        torch.cuda.synchronize()
        kept = sum(rr[k].numel() * rr[k].element_size() for k in ("ws", "colmax", "rank"))
        kept += rr["packed"].buf.numel()
        transient = torch.cuda.max_memory_allocated() - base - kept
        assert transient < whole_packed, (transient, whole_packed)
        c, m, i = ev.evaluate(qf, s.q_pids, s.q_camids, return_distmat=True)
        parts = [torch.empty((qf.shape[0], b - a), device="cuda") for a, b in bounds]
        dist.all_gather(parts, i["distmat"].contiguous())
        d = torch.cat(parts, 1)
        assert torch.equal(d.view(torch.int32), i0["distmat"].view(torch.int32)), exchange
        assert np.array_equal(c, c0) and m == m0 and i["mINP"] == i0["mINP"], exchange
        assert torch.equal(i["ap"], i0["ap"]) and torch.equal(i["first"], i0["first"]), exchange
        idx, val = ev.ranked_lists(qf, s.q_pids, s.q_camids, k=20)
        assert torch.equal(idx, r0[0]) and torch.equal(val, r0[1]), exchange
    dist.barrier()
    out[rank] = True
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_without_the_whole_gallery():
    """Two GPUs, unaligned slices, both exchanges: distmat, cmc, mAP, mINP, ap, first and ranked lists equal one GPU's,
    and what a rank's prepare allocates beyond the state it keeps stays below the packed size of the whole gallery."""
    import torch.multiprocessing as mp
    world = 2
    out = mp.Manager().dict()
    mp.spawn(_multi_gpu_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert dict(out) == {r: True for r in range(world)}
