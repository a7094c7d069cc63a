"""GNN re-ranking shared by the ranks of a query_group (RetrievalEvaluator(rerank="gnn", query_group=...)), at every world
size of 1, 2, 4 and 8 the box has: one process per GPU over NCCL, every rank holding the whole gallery.

Sets: the 10 000 x 140 000 x 256 set of test_gpu_gnn_stream.py::test_beyond_both_dense_limits (k1 = 26, k2 = 7), and
with --large a set near the N limit (48 000 x 1 000 000 x 256, generated on the device from a seed).

Per rank, from the evaluator's CUDA-event marks (IEEE_B200_TRACE; an interval is charged to the mark that ends it) of
one evaluate() after a warm-up evaluate() of another query tensor:
  prepare  neighbours (with the query pack), each exchange, the symbolic phase, the sizes (the host round trip), each
           numeric step, the CSC
  blocks   the GNN similarity of the rank's query blocks, the rank stages, the exchange of per-query results, the reduce
and the peak of torch.cuda.max_memory_allocated over that evaluate(), A's nnz, and whether cmc, mAP, mINP, ap and first
equal an evaluator without query_group (run first, in the rank-0 process of world size 1, and timed the same way: the
one-GPU streamed form's stage split).

    python profiles/gnn_shard_probe.py [--worlds 1,2,4,8] [--large] [--out FILE]
"""
import argparse
import os
import socket
import subprocess
import sys
import tempfile

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["IEEE_B200_TRACE"] = "1"
from ieee_b200 import engine                                                 # noqa: E402
from ieee_b200.engine import RetrievalEvaluator, rerank_owned                # noqa: E402
from ieee_b200.testing import make_retrieval_set                              # noqa: E402

STAGES = ["neighbours", "exchange rank,S", "symbolic", "exchange counts", "sizes", "numeric 0", "exchange 0", "numeric 1",
          "exchange 1", "numeric 2", "exchange 2", "numeric 3", "exchange A gallery rows", "CSC", "exchange CSC",
          "numeric (one call)", "blocks: similarity", "blocks: rank stages", "exchange results", "reduce"]
MARKS = {"GNN neighbours": "neighbours", "GNN exchange: rank, S": "exchange rank,S", "GNN symbolic phase": "symbolic",
         "GNN exchange: counts": "exchange counts", "GNN sizes": "sizes", "GNN exchange: gallery rows of A": "exchange A gallery rows",
         "GNN CSC": "CSC", "GNN exchange: CSC": "exchange CSC", "GNN numeric phase": "numeric (one call)",
         "  GNN similarity": "blocks: similarity", "rank stages done": "exchange results", "reduce done": "reduce"}


def unit(t):
    return torch.nn.functional.normalize(t.float(), dim=1)


def make_set(name):
    if name == "10000x140000x256":
        s = make_retrieval_set(10000, 140000, 5000, 6, dim=256, sigma=2.75, seed=7)
        return unit(s.qf).cuda(), unit(s.gf).cuda(), s.q_pids, s.g_pids, s.q_camids, s.g_camids
    Q, G, D, ids = 48000, 1000000, 256, 20000                   # near N = 2^20, generated on the device
    gen = torch.Generator(device="cuda").manual_seed(1)
    centers = torch.randn(ids, D, generator=gen, device="cuda")
    q_ids = torch.randint(0, ids, (Q,), generator=gen, device="cuda")
    g_ids = torch.randint(0, ids, (G,), generator=gen, device="cuda")
    qf = unit(centers[q_ids] + 2.75 * torch.randn(Q, D, generator=gen, device="cuda"))
    gf = torch.empty(G, D, device="cuda")
    for s in range(0, G, 100000):
        e = min(G, s + 100000)
        gf[s:e] = unit(centers[g_ids[s:e]] + 2.75 * torch.randn(e - s, D, generator=gen, device="cuda"))
    cams = torch.randint(0, 6, (Q + G,), generator=gen, device="cuda").cpu().numpy()
    return qf, gf, q_ids.cpu().numpy(), g_ids.cpu().numpy(), cams[:Q], cams[Q:]


def categorise(marks):
    """ms per stage from [(name, event)]."""
    t = {k: 0.0 for k in STAGES}
    for (_, e0), (name, e1) in zip(marks, marks[1:]):
        ms = e0.elapsed_time(e1)
        if name in MARKS:
            t[MARKS[name]] += ms
        elif name.startswith("GNN numeric step"):
            t["numeric " + name.split()[-1]] += ms
        elif name.startswith("GNN exchange after step"):
            t["exchange " + name.split()[-1]] += ms
        elif name.startswith("  "):
            t["blocks: rank stages"] += ms
    return {k: v for k, v in t.items() if v > 0}


def timed_evaluate(ev, qf, q_ids, q_cams):
    """evaluate() after a warm-up of another query tensor: (results, stage split, peak bytes)."""
    captured = []

    def keep_marks():                                                    # instead of printing them
        captured.append(list(engine.TRACE.marks))
        engine.TRACE.marks = []
    engine.TRACE.report = keep_marks
    ev.evaluate(qf.clone(), q_ids, q_cams)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    engine.TRACE.marks = []
    out = ev.evaluate(qf, q_ids, q_cams)
    torch.cuda.synchronize()
    return out, categorise([(n, e) for n, e, _ in captured[-1]]), torch.cuda.max_memory_allocated()


def fmt(split):
    return "  ".join("%s %.1f" % kv for kv in split.items()) + "  (ms) total %.1f ms" % sum(split.values())


def worker(rank, world, port, name, ref_path, out_path):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    qf, gf, q_ids, g_ids, q_cams, g_cams = make_set(name)
    Q, G = qf.shape[0], gf.shape[0]
    if world == 1 and rank == 0 and not os.path.exists(ref_path):
        ref = RetrievalEvaluator(gf, g_ids, g_cams, rerank="gnn", block_bytes=1 << 30)
        (c, m, i), split, peak = timed_evaluate(ref, qf, q_ids, q_cams)
        nnz = ref._rr["a_col"].numel()
        np.savez(ref_path, cmc=c, mAP=m, mINP=i["mINP"], ap=i["ap"].cpu().numpy(), first=i["first"].cpu().numpy())
        with open(out_path, "a") as f:
            f.write("%s  no query_group (one-GPU streamed form)  %s | nnz(A) %d | peak %.2f GB\n" % (name, fmt(split), nnz, peak / 1e9))
        del ref
    ev = RetrievalEvaluator(gf, g_ids, g_cams, rerank="gnn", block_bytes=1 << 30, query_group=dist.group.WORLD)
    (cmc, mAP, info), split, peak = timed_evaluate(ev, qf, q_ids, q_cams)
    ref = np.load(ref_path)
    same = (np.array_equal(cmc, ref["cmc"]) and mAP == float(ref["mAP"]) and info["mINP"] == float(ref["mINP"])
            and np.array_equal(info["ap"].cpu().numpy(), ref["ap"]) and np.array_equal(info["first"].cpu().numpy(), ref["first"]))
    q0, q1, g0, g1 = rerank_owned(Q, G, world, rank)
    with open(out_path, "a") as f:
        f.write("%s  query_group world %d rank %d (queries [%d, %d), gallery rows [%d, %d))  %s | nnz(A) %d | peak %.2f GB | "
                "bit-identical to no query_group: %s\n" % (name, world, rank, q0, q1, g0, g1, fmt(split), ev._rr["a_col"].numel(),
                                                            peak / 1e9, "yes" if same else "NO"))
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--large", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch.multiprocessing as mp
    n_gpu = torch.cuda.device_count()
    asked = list(map(int, a.worlds.split(",")))
    worlds = sorted(set([1] + [w for w in asked if w <= n_gpu]))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# gnn_shard_probe, k1 = 26, k2 = 7, block_bytes = 1 GiB, on %s (name, power limit, max SM clock); %d GPU(s) in "
             "the box" % (gpu[0] if gpu else "?", n_gpu)]
    lines += ["# world %d: not measured (the box has %d GPU(s))" % (w, n_gpu) for w in asked if w not in worlds]
    names = ["10000x140000x256"] + (["48000x1000000x256"] if a.large else [])
    lines += ["# 48000x1000000x256: not measured"] if not a.large else []
    lines.append("")
    with tempfile.TemporaryDirectory() as tmp:
        for name in names:
            ref_path, out_path = os.path.join(tmp, name + ".npz"), os.path.join(tmp, name + ".txt")
            for world in worlds:
                with socket.socket() as sk:
                    sk.bind(("127.0.0.1", 0))
                    port = sk.getsockname()[1]
                mp.spawn(worker, args=(world, port, name, ref_path, out_path), nprocs=world, join=True)
            lines += open(out_path).read().splitlines()
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
