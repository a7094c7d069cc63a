"""GNN re-ranking, dense (gnn_reranking_distmat: -(X_u X_u^T), ieee_gnn_rerank, A[:Q] A[Q:]^T, then evaluate_device)
against streamed (RetrievalEvaluator(rerank="gnn"): neighbours from row strips, symbolic and numeric phases, one
ieee_gnn_stream_block per query block), on one GPU, k1 = 26, k2 = 7, L2-normalised float32 features, f16x3:

  C3      RGBNT201-shaped, Q = G = 836 (query set == gallery set), D = 2304
  market  Market-1501-shaped, 3368 x 15913, D = 2304
  large   10 000 x 140 000, D = 256: N = 150 000 is past the dense propagation's 65 535 rows, and the dense form
          would need about 12 N^2 = 270 GB

Times are device-synchronised wall times, median of --reps runs after one warm-up run: the dense pipeline, a whole
evaluate() of a fresh query set (state + block loop), and the state alone.  Stage split from one torch.profiler run
(kernel time, summed by stage in launch order): strips (contractions, top-k, squares), symbolic (transposes of the
neighbour lists, counts, offsets), numeric (B = A + A^T, propagation and normalisation, transposes, the gallery CSC),
per-block similarity (gnn_block_kernel) and rank stages.  Peak memory is torch.cuda.max_memory_allocated over one
whole run from nothing but the features.  nnz/row and in-degree are those of the final A.

    python profiles/gnn_stream_probe.py [--sets c3,market,large] [--reps 3] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ieee_b200.engine import DEFAULT_BLOCK_BYTES, RetrievalEvaluator                             # noqa: E402
from ieee_b200.metrics.rank import evaluate_device                                              # noqa: E402
from ieee_b200.testing import market1501_shaped, rgbnt201_shaped                                # noqa: E402
from ieee_b200.utils.gnn_reranking import gnn_reranking_distmat                                  # noqa: E402

K1, K2 = 26, 7


def large_set(Q=10000, G=140000, D=256, ids=5000, sigma=2.75, seed=0):
    """Identity-clustered features generated on the device (seeded), L2-normalised."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    centers = torch.randn(ids, D, generator=gen, device="cuda")
    q_ids = torch.randint(0, ids, (Q,), generator=gen, device="cuda")
    g_ids = torch.randint(0, ids, (G,), generator=gen, device="cuda")
    qf = centers[q_ids] + sigma * torch.randn(Q, D, generator=gen, device="cuda")
    gf = centers[g_ids] + sigma * torch.randn(G, D, generator=gen, device="cuda")
    q_cams = torch.randint(0, 6, (Q,), generator=gen, device="cuda")
    g_cams = torch.randint(0, 6, (G,), generator=gen, device="cuda")
    return (unit(qf), unit(gf), q_ids.cpu().numpy(), g_ids.cpu().numpy(), q_cams.cpu().numpy(), g_cams.cpu().numpy())


def unit(x):
    return torch.nn.functional.normalize(x.float(), dim=1)


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts) * 1e3, out


def peak_of(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 2**30


def stage_split(ev, qf, q_pids, q_camids):
    from torch.profiler import ProfilerActivity, profile
    ev._rr = None
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ev.evaluate(qf, q_pids, q_camids)
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
    out = {"strips": 0.0, "symbolic": 0.0, "numeric": 0.0, "block similarity": 0.0, "rank stages": 0.0}
    stage = "strips"
    for e in kernels:
        n = e.name
        us = getattr(e, "device_time_total", None)
        us = e.cuda_time_total if us is None else us
        if stage == "strips" and any(k in n for k in ("gnn_iota", "gnn_rank_count")):
            stage = "symbolic"
        elif stage == "symbolic" and "gnn_sum" in n:
            stage = "numeric"
        elif stage != "blocks" and "gnn_block" in n:
            stage = "blocks"
        if stage == "blocks":
            out["block similarity" if "gnn_block" in n else "rank stages"] += us / 1e3
        else:
            out[stage] += us / 1e3
    return out


def probe(name, qf, gf, q_pids, g_pids, q_camids, g_camids, reps, lines):
    Q, G, D = qf.shape[0], gf.shape[0], qf.shape[1]
    N = Q + G
    lines.append("== %s: Q = %d, G = %d, N = %d, D = %d, k1 = %d, k2 = %d, f16x3, block_bytes = %d GiB"
                 % (name, Q, G, N, D, K1, K2, DEFAULT_BLOCK_BYTES >> 30))
    dense_ms = None
    if N <= 65535 and 12 * N * N < (150 << 30):
        def dense():
            out = gnn_reranking_distmat(qf, gf, K1, K2)
            _, summary, _ = evaluate_device(out, q_pids, g_pids, q_camids, g_camids, 20)
            return summary.mAP
        dense_ms, dense_map = timed(dense, reps)
        dense_peak = peak_of(dense)
        lines.append("dense     total %10.1f ms   peak %7.2f GiB   mAP %.4f" % (dense_ms, dense_peak, dense_map))
    else:
        lines.append("dense     not run: N = %d rows (the propagation launch takes at most 65 535) and about %.0f GB "
                     "(12 N^2 bytes)" % (N, 12 * N * N / 1e9))
    ev = RetrievalEvaluator(gf, g_pids, g_camids, rerank="gnn", k1=K1, k2=K2)

    def streamed():
        ev._rr = None                      # a fresh query set: state + blocks
        return ev.evaluate(qf, q_pids, q_camids)[1]

    def state_only():
        ev._rr = None
        ev._rerank_prepare(qf)
    st_ms, st_map = timed(streamed, reps)
    prep_ms, _ = timed(state_only, reps)
    rr = ev._rr
    deg = rr["a_ptr"].diff().double()
    indeg = torch.bincount(rr["a_col"].long(), minlength=N).max().item()
    nnz_line = "A: nnz %d, nnz/row mean %.0f max %d, max in-degree %d; gallery CSC nnz %d" % (
        rr["a_col"].numel(), deg.mean().item(), int(deg.max().item()), indeg, rr["g_row"].numel())
    ev._rr = ev._block = None
    st_peak = peak_of(lambda: RetrievalEvaluator(gf, g_pids, g_camids, rerank="gnn", k1=K1, k2=K2).evaluate(qf, q_pids, q_camids))
    lines.append("streamed  total %10.1f ms   peak %7.2f GiB   mAP %.4f   (state %.1f ms, block loop %.1f ms)"
                 % (st_ms, st_peak, st_map, prep_ms, st_ms - prep_ms))
    if dense_ms is not None:
        lines.append("streamed / dense: %.2fx   |mAP difference| %.2e" % (st_ms / dense_ms, abs(st_map - dense_map)))
    lines.append(nnz_line)
    split = stage_split(ev, qf, q_pids, q_camids)
    lines.append("stage split (kernel time, ms): " + ", ".join("%s %.1f" % kv for kv in split.items()))
    lines.append("")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", default="c3,market,large")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# gnn_stream_probe on %s (name, power limit, max SM clock)" % (gpu[torch.cuda.current_device()] if gpu else "?"), ""]
    for name in a.sets.split(","):
        if name == "c3":
            s = rgbnt201_shaped()
        elif name == "market":
            s = market1501_shaped()
        if name in ("c3", "market"):
            args = (unit(s.qf).cuda(), unit(s.gf).cuda(), s.q_pids, s.g_pids, s.q_camids, s.g_camids)
        else:
            args = large_set()
        probe(name, *args, reps=a.reps if name != "large" else 1, lines=lines)
        print("\n".join(lines[-7:]), flush=True)
    text = "\n".join(lines) + "\n"
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
