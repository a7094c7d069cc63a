"""k-reciprocal re-ranking over a gallery sharded across the GPUs of one box (RetrievalEvaluator(group=..., rerank=True)),
20 000 queries x 300 000 gallery rows x 2304, at every world size of 1, 2, 4 and 8 the box has: one process per GPU
over NCCL, the gallery split with shard_bounds.

Per rank, from the evaluator's CUDA-event marks (IEEE_B200_TRACE; an interval is charged to the mark that ends it) of
one evaluate() after a warm-up evaluate() of another query tensor:
  prepare  range (the rank's gallery range packed, and the query pack before it), pass 0 (colmax and rank, with the
           per-strip exchanges: strip rows, colmax, neighbour lists), pass 1 (V, with the per-strip exchanges: strip
           rows, V's values), finish (query expansion and inverted index of the rank's slice)
  blocks   per query block: contraction against the slice, re-ranking blend, rank stages (gather, exchanges, counts)
and the peak of torch.cuda.max_memory_allocated over that evaluate().  Every rank compares its cmc, mAP, ap and first
with a one-GPU rerank=True evaluator on the whole gallery, run first in the rank-0 process of world size 1 and saved.

    python profiles/rerank_shard_probe.py [--worlds 1,2,4,8] [--q 20000] [--g 300000] [--out FILE]
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
from ieee_b200.engine import RetrievalEvaluator, shard_bounds                # noqa: E402

PREPARE = [("range", "re-ranking: gallery range"), ("pass 0", "re-ranking: pass 0"), ("pass 1", "re-ranking: pass 1"),
           ("finish", "re-ranking state prepared")]


def make_set(Q, G, D=2304, ids=3000, sigma=3.0, seed=0):
    """Identity-clustered features, generated on the device from a seed (the same on every rank)."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    centers = torch.randn(ids, D, generator=gen, device="cuda")
    q_ids = torch.randint(0, ids, (Q,), generator=gen, device="cuda")
    g_ids = torch.randint(0, ids, (G,), generator=gen, device="cuda")
    qf = torch.relu(centers[q_ids] + sigma * torch.randn(Q, D, generator=gen, device="cuda"))
    gf = torch.empty(G, D, device="cuda")
    for s in range(0, G, 50000):
        e = min(G, s + 50000)
        gf[s:e] = torch.relu(centers[g_ids[s:e]] + sigma * torch.randn(e - s, D, generator=gen, device="cuda"))
    cams = torch.randint(0, 6, (Q + G,), generator=gen, device="cuda").cpu().numpy()
    return qf, gf, q_ids.cpu().numpy(), g_ids.cpu().numpy(), cams[:Q], cams[Q:]


def categorise(marks):
    """(prepare split in ms, per-block contraction / blend / rank in ms, number of blocks) from [(name, event)]."""
    prep = {k: 0.0 for k, _ in PREPARE}
    blocks = {"contraction": 0.0, "blend": 0.0, "rank": 0.0}
    n_blocks = 0
    for (_, e0), (name, e1) in zip(marks, marks[1:]):
        ms = e0.elapsed_time(e1)
        hit = [k for k, prefix in PREPARE if name.startswith(prefix)]
        if hit:
            prep[hit[0]] += ms
        elif "chunk" in name:
            blocks["contraction"] += ms
            n_blocks += 1
        elif "re-ranking blend" in name:
            blocks["blend"] += ms
        elif name.startswith("  ") or name in ("rank stages done", "reduce done"):
            blocks["rank"] += ms
    return prep, {k: v / max(n_blocks, 1) for k, v in blocks.items()}, n_blocks


def worker(rank, world, port, Q, G, ref_path, out_path):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    qf, gf, q_ids, g_ids, q_cams, g_cams = make_set(Q, G)
    if world == 1 and rank == 0 and not os.path.exists(ref_path):
        ref = RetrievalEvaluator(gf, g_ids, g_cams, rerank=True)
        c, m, i = ref.evaluate(qf, q_ids, q_cams)
        np.savez(ref_path, cmc=c, mAP=m, ap=i["ap"].cpu().numpy(), first=i["first"].cpu().numpy())
        del ref
        engine.TRACE.marks = []
    g0, g1 = shard_bounds(G, world, rank)
    ev = RetrievalEvaluator(gf[g0:g1].contiguous(), g_ids[g0:g1], g_cams[g0:g1], rerank=True, group=dist.group.WORLD,
                            g_offset=g0, g_total=G)
    del gf
    captured = []

    def keep_marks():                                                    # instead of printing them
        captured.append(list(engine.TRACE.marks))
        engine.TRACE.marks = []
    engine.TRACE.report = keep_marks
    ev.evaluate(qf.clone(), q_ids, q_cams)                                # warm-up, its own prepare
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    engine.TRACE.marks = []
    cmc, mAP, info = ev.evaluate(qf, q_ids, q_cams)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    prep, blk, n_blocks = categorise([(n, e) for n, e, _ in captured[-1]])
    ref = np.load(ref_path)
    same = (np.array_equal(cmc, ref["cmc"]) and mAP == float(ref["mAP"]) and np.array_equal(info["ap"].cpu().numpy(), ref["ap"])
            and np.array_equal(info["first"].cpu().numpy(), ref["first"]))
    line = ("world %d rank %d  slice %7d rows  prepare %s  total %.1f ms | %d blocks, per block: contraction %.2f ms, "
            "blend %.2f ms, rank %.2f ms | peak %.2f GB | bit-identical to one GPU: %s"
            % (world, rank, g1 - g0, "  ".join("%s %.1f ms" % kv for kv in prep.items()), sum(prep.values()), n_blocks,
               blk["contraction"], blk["blend"], blk["rank"], peak / 1e9, "yes" if same else "NO"))
    with open(out_path, "a") as f:
        f.write(line + "\n")
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--q", type=int, default=20000)
    ap.add_argument("--g", type=int, default=300000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch.multiprocessing as mp
    n_gpu = torch.cuda.device_count()
    worlds = [w for w in map(int, a.worlds.split(",")) if w <= n_gpu]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# rerank_shard_probe, %d x %d x 2304, on %s (name, power limit, max SM clock); %d GPU(s) in the box"
             % (a.q, a.g, gpu[0] if gpu else "?", n_gpu), ""]
    with tempfile.TemporaryDirectory() as tmp:
        ref_path, out_path = os.path.join(tmp, "ref.npz"), os.path.join(tmp, "out.txt")
        for world in sorted(set([1] + worlds)):
            with socket.socket() as sk:
                sk.bind(("127.0.0.1", 0))
                port = sk.getsockname()[1]
            mp.spawn(worker, args=(world, port, a.q, a.g, ref_path, out_path), nprocs=world, join=True)
        lines += sorted(open(out_path).read().splitlines())
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
