"""k-reciprocal re-ranking, dense (ieee_rerank on qg, qq, gg) against streamed (RetrievalEvaluator(rerank=True):
ieee_rerank_stream_prepare + one ieee_rerank_stream_block per query block), on one GPU:

  C3      RGBNT201-shaped, Q = G = 836 (query set == gallery set), D = 2304
  market  Market-1501-shaped, 3368 x 15913, D = 2304
  large   20 000 x 300 000, D = 2304: the dense path would need 8 N^2 = 819 GB

Times are device-synchronised wall times, median of --reps runs after one warm-up run:
  dense     three contractions (qg, qq, gg) + ieee_rerank + evaluate_device
  streamed  a whole evaluate() of a fresh query set (prepare + block loop), and its prepare alone
Stage split of the streamed form from one torch.profiler run (kernel time only, summed by stage): pass 1
(contractions, column maxima, orig rows, top-k), pass 2 (contractions, orig rows, weights), sparse stages (membership,
query expansion, inverted index), and per query block its contraction, the re-ranking blend and the rank stages.  Peak
memory is torch.cuda.max_memory_allocated over one whole run from nothing but the features: the dense arm's packing,
three matrices, workspace and rank buffers; the streamed arm's evaluator (gallery packing, re-ranking state, strips,
distance block, blend accumulators, rank buffers).

    python profiles/rerank_stream_probe.py [--sets c3,market,large] [--reps 3] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ieee_b200.engine import DEFAULT_BLOCK_BYTES, PackedFeatures, RetrievalEvaluator, packed_distmat   # noqa: E402
from ieee_b200.metrics.rank import evaluate_device                                                   # noqa: E402
from ieee_b200.testing import market1501_shaped, rgbnt201_shaped                                     # noqa: E402
from ieee_b200.utils.rerank import re_ranking_device                                                 # noqa: E402

DENSE_LIMIT = 150 << 30        # bytes of dense state this probe allows itself on a 180 GB card


def large_set(Q=20000, G=300000, D=2304, ids=3000, sigma=3.0, seed=0):
    """Identity-clustered features generated on the device (seeded), as ieee_b200.testing builds them on the host."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    centers = torch.randn(ids, D, generator=gen, device="cuda")
    q_ids = torch.randint(0, ids, (Q,), generator=gen, device="cuda")
    g_ids = torch.randint(0, ids, (G,), generator=gen, device="cuda")
    qf = torch.relu(centers[q_ids] + sigma * torch.randn(Q, D, generator=gen, device="cuda"))
    gf = torch.empty(G, D, device="cuda")
    for s in range(0, G, 50000):
        e = min(G, s + 50000)
        gf[s:e] = torch.relu(centers[g_ids[s:e]] + sigma * torch.randn(e - s, D, generator=gen, device="cuda"))
    q_cams = torch.randint(0, 6, (Q,), generator=gen, device="cuda")
    g_cams = torch.randint(0, 6, (G,), generator=gen, device="cuda")
    return qf, gf, q_ids.cpu().numpy(), g_ids.cpu().numpy(), q_cams.cpu().numpy(), g_cams.cpu().numpy()


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
    """Kernel time per stage of one evaluate() with a fresh re-ranking state.  Kernels are taken in launch order:
    everything up to the membership kernel is pass 1 (the query set's packing included), from there to the query
    expansion pass 2, the sparse kernels themselves are 'sparse', and after them come the query blocks: packing and
    contraction, the blend (rr_jaccard_kernel) and the rank stages (everything else)."""
    from torch.profiler import ProfilerActivity, profile
    ev._rr = None
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ev.evaluate(qf, q_pids, q_camids)
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
    out = {"pass 1": 0.0, "pass 2": 0.0, "sparse": 0.0, "block contraction": 0.0, "blend": 0.0, "rank stages": 0.0}
    stage = "pass 1"
    for e in kernels:
        n = e.name
        us = getattr(e, "device_time_total", None)
        us = e.cuda_time_total if us is None else us
        if "rr_krecip" in n:
            out["sparse"] += us / 1e3
            stage = "pass 2"
        elif any(k in n for k in ("rr_expand", "rr_col_count", "rr_scan", "rr_col_fill")):
            out["sparse"] += us / 1e3
            stage = "blocks"
        elif stage == "blocks":
            part = "blend" if "rr_jaccard" in n else "block contraction" if ("distmat" in n or "pack_rows" in n) else "rank stages"
            out[part] += us / 1e3
        else:
            out[stage] += us / 1e3
    return out


def probe(name, qf, gf, q_pids, g_pids, q_camids, g_camids, reps, lines):
    Q, G, D = qf.shape[0], gf.shape[0], qf.shape[1]
    N = Q + G
    lines.append("== %s: Q = %d, G = %d, N = %d, D = %d, k1 = 20, k2 = 6, lambda = 0.3, f16x3, block_bytes = %d GiB"
                 % (name, Q, G, N, D, DEFAULT_BLOCK_BYTES >> 30))
    dense_bytes = 8 * N * N
    dense_ms = None
    ev = RetrievalEvaluator(gf, g_pids, g_camids, rerank=True)
    ev.evaluate(qf, q_pids, q_camids)        # fixes the centre (from the query set) both forms pack with
    if dense_bytes <= DENSE_LIMIT:
        def dense():
            qpk = PackedFeatures(qf, "euclidean", False, "f16x3", ev.center)
            gpk = PackedFeatures(gf, "euclidean", False, "f16x3", ev.center)
            qg = packed_distmat(qpk, gpk, torch.empty((Q, G), device="cuda"))
            qq = packed_distmat(qpk, qpk, torch.empty((Q, Q), device="cuda"))
            gg = packed_distmat(gpk, gpk, torch.empty((G, G), device="cuda"))
            out = re_ranking_device(qg, qq, gg)
            cmc, summary, _ = evaluate_device(out, q_pids, g_pids, q_camids, g_camids, 20)
            return summary.mAP
        dense_ms, dense_map = timed(dense, reps)
        dense_peak = peak_of(dense)
        lines.append("dense     total %10.1f ms   peak %7.2f GiB   mAP %.4f" % (dense_ms, dense_peak, dense_map))
    else:
        lines.append("dense     not run: needs about %.0f GB (8 N^2 bytes) of HBM" % (dense_bytes / 1e9))

    def streamed():
        ev._rr = None                      # a fresh query set: prepare + blocks
        return ev.evaluate(qf, q_pids, q_camids)[1]

    def prepare_only():
        ev._rr = None
        ev._rerank_prepare(qf)
    st_ms, st_map = timed(streamed, reps)
    prep_ms, _ = timed(prepare_only, reps)
    ev._rr = ev._block = ev._rr_scratch = None
    st_peak = peak_of(lambda: RetrievalEvaluator(gf, g_pids, g_camids, rerank=True).evaluate(qf, q_pids, q_camids))
    lines.append("streamed  total %10.1f ms   peak %7.2f GiB   mAP %.4f   (prepare %.1f ms, block loop %.1f ms)"
                 % (st_ms, st_peak, st_map, prep_ms, st_ms - prep_ms))
    if dense_ms is not None:
        lines.append("streamed / dense: %.2fx   mAP equal: %s" % (st_ms / dense_ms, st_map == dense_map))
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
    lines = ["# rerank_stream_probe on %s (name, power limit, max SM clock)" % (gpu[torch.cuda.current_device()] if gpu else "?"), ""]
    for name in a.sets.split(","):
        if name == "c3":
            s = rgbnt201_shaped()
            args = (s.qf.cuda(), s.gf.cuda(), s.q_pids, s.g_pids, s.q_camids, s.g_camids)
        elif name == "market":
            s = market1501_shaped()
            args = (s.qf.cuda(), s.gf.cuda(), s.q_pids, s.g_pids, s.q_camids, s.g_camids)
        else:
            args = large_set()
        probe(name, *args, reps=a.reps if name != "large" else 1, lines=lines)
        print("\n".join(lines[-6:]), flush=True)
    text = "\n".join(lines) + "\n"
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
