#!/usr/bin/env python
"""bench.py -- queries/sec of the retrieval hot path (distmat + rank + CMC/mAP) on B200.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the reference's CPU path (torch CPU distance + Cython rank)
    python bench.py ... --dump-outputs DIR      # also write the last timed step's results as DIR/<name>.npy

One "step" = one pass of the hot path over one synthetic evaluation set: features + labels in,
(cmc, mAP) on the host out.  Workload (BASELINE.json configs[1]): Market1501-multimodal-shaped,
3368 queries x 15913 gallery x 2304-d float32, euclidean, max_rank 20.  With N GPUs the gallery is
sharded by rows (contiguous slices), every rank sees all queries, and the query set grows to 3368*N so
that per-GPU work stays fixed ("weak"): relevant lists and partial counts are exchanged as stores into
NVLink peer memory from inside the rank kernels (IEEE_B200_EXCHANGE=nccl: all-gather + all-reduce).
Prints ONE JSON line on rank 0.

Besides the timed headline the line carries, on rank 0:
  result.parity   sharded == single-GPU (bit for bit) and a 512-query subsample against the CPU oracle / the
                  compiled reference (distances within 1e-4 relative + the reference's own floor, CMC bit-exact,
                  mAP within 1e-6 on identical distances)
  extras (N = 1)  config C1 (real-model fixture), C2 with cosine, C3 (k-reciprocal re-ranking) and one C4-shaped gallery
                  shard (8192 queries x 125 000 rows): time, roofline fraction, parity and the CPU path beside each.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

Q_BASE, G_TOTAL, DIM, PIDS, CAMS, MAX_RANK = 3368, 15913, 2304, 751, 6, 20
METRIC_NAME = "queries/sec (distmat+rank+CMC/mAP)"
REF_SAMPLE_Q = 512          # query rows the CPU arms and the parity check take from the workload


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def make_workload(n_gpus: int):
    from ieee_b200.testing import market1501_shaped
    return market1501_shaped(seed=1, num_q=Q_BASE * n_gpus)


def bench_config(n_gpus: int) -> dict:
    """The `config` object: the same for our arm and the reference arm at a given N."""
    n = max(1, n_gpus)
    return {"workload": f"market1501_shaped Q={Q_BASE * n} G={G_TOTAL} D={DIM} euclidean max_rank={MAX_RANK}",
            "gallery_sharding": f"{n} contiguous row shards", "queries": "replicated on every rank",
            "timing": "cyclic GC off inside the timed loops of both arms (as timeit does)",
            "l2": "per-step working set (features 178 MB + packed 178 MB + distmat 214 MB per GPU) exceeds the 126 MB L2; "
                  "stage timings flush L2 with a 256 MB write between repetitions"}


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region, read through NVML (rank 0 only).

    mode "thread" (default): a sampling thread reads every few milliseconds while the timing loop runs.  The NVML calls
    are C calls made through ctypes, so the thread holds the GIL only for the few microseconds between them -- the
    loop being timed never waits for a reading.  (Readings made BY the loop cost ~40 us each on one GPU but 2 - 40 ms
    each once several ranks share the node, and rank 0 being late stalls every rank at the next hand-over: N = 4
    measured 6.6 ms per step that way; an `nvidia-smi -lms` child process slowed a 2-GPU step from 0.9 to 3.4 ms.)
    mode "loop": readings by the timing loop at steps K/4, K/2, 3K/4.  mode "after": no reading inside the timed
    region; K more steps of the same load follow it at once and are sampled by the loop (their time is not used)."""

    def __init__(self, index: int, enabled: bool = True, mode: str | None = None):
        self.samples, self.reasons, self.max_mhz, self.nv = [], set(), None, None
        self.mode = mode or os.environ.get("IEEE_BENCH_CLOCKS", "thread")
        self._thread, self._stop = None, None
        if not enabled:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.names = {"hw_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                          "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                          "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                          "sw_power_cap": getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            # the first NVML queries of a process take tens of milliseconds: pay that here, outside the timed region
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        except Exception:
            self.nv = None

    def sample(self):
        if self.nv is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for k, bit in self.names.items():
                if mask & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def arm(self):
        """Before the warm-up: the sampling thread is created here (thread start-up costs ~0.1 ms) and parks on `go`."""
        if self.nv is None or self.mode != "thread":
            return
        import threading
        self._stop, self._go = threading.Event(), threading.Event()

        def run():
            self._go.wait()
            while not self._stop.wait(0.004):        # first reading 4 ms into the region, then every 4 ms
                self.sample()
            if not self.samples:
                self.sample()                        # a region shorter than one interval: one reading at its end

        self._thread = threading.Thread(target=run, daemon=True)
        self._thread.start()

    def start(self):
        """Right after the start event is recorded: releases the sampling thread (an Event.set, microseconds)."""
        if self._thread is not None:
            self._go.set()

    def stop(self):
        """Called right after the stop event is recorded (the GPU is still working through the queue)."""
        if self._thread is not None:
            self._stop.set()
            self._go.set()
            self._thread.join()
            self._thread = None

    def result(self):
        how = {"thread": "NVML readings by a sampling thread (every ~4 ms) while the timed region runs",
               "loop": "NVML readings taken by the timing loop between steps of the timed region",
               "after": "NVML readings between steps of a second pass of the same K steps that follows the timed region at once "
                        "(no reading inside the timed region itself)"}[self.mode]
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "how": how}


# ------------------------------------------------------------------------------------------------------
# the reference arm / CPU baselines: the reference's own CPU path on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_reference_path():
    """Returns (kind, module-like with compute_distance_matrix / evaluate_cy / re_ranking): oracle/_ref (the
    reference's files, compiled) when present, else the oracle port."""
    from oracle import ref, restatement
    if ref.available():
        return "reference", ref
    port = type("Port", (), {})()
    port.compute_distance_matrix = restatement.compute_distance_matrix
    port.evaluate_cy = lambda d, qp, gp, qc, gc, k: restatement.evaluate_rank(d, qp, gp, qc, gc, max_rank=k)
    port.re_ranking = restatement.re_ranking
    return "port", port


def time_cpu_path(qf, gf, q_pids, g_pids, q_camids, g_camids, metric, steps, warmup):
    """torch CPU distance (distance.py:59-80) + Cython rank (rank_cy.pyx:156-243); returns (s per pass, kind, cores)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kind, ref = cpu_reference_path()
    times = []
    gc_was_on = gc.isenabled()
    gc.collect()
    gc.disable()                 # same rule as our arm's timed loop
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        d = ref.compute_distance_matrix(qf, gf, metric).numpy()
        ref.evaluate_cy(d, q_pids, g_pids, q_camids, g_camids, MAX_RANK)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    if gc_was_on:
        gc.enable()
    return sum(times) / len(times), kind, cores


def cpu_sample_text(sample_q, cores):
    return (f"each step: first {sample_q} queries of the workload x full {G_TOTAL}-row gallery; torch CPU distance "
            f"({cores} threads) + rank_cy.evaluate_cy (single-threaded by construction)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = max(1, args.gpus)
    ws = make_workload(n)
    sq = REF_SAMPLE_Q
    sec, kind, cores = time_cpu_path(ws.qf[:sq], ws.gf, ws.q_pids[:sq], ws.g_pids, ws.q_camids[:sq], ws.g_camids, "euclidean",
                                     args.steps, args.warmup)
    qps = sq / sec
    line = {
        "impl": "reference", "metric": METRIC_NAME, "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": bench_config(n),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": kind, "sample": cpu_sample_text(sq, cores)},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# parity, recorded in the JSON line
# ------------------------------------------------------------------------------------------------------
def distance_ratio(d, d_ref, a, b, atol_scale=8e-7, rtol=1e-4, chunk=256):
    """max over all pairs of |d - d_ref| / (rtol |d_ref| + atol_scale (|a|^2 + |b|^2)): <= 1 is parity (north_star's
    1e-4 relative plus twice the cancellation floor the reference's own fp32 GEMM sits on)."""
    nb = (b.double() ** 2).sum(1).numpy()
    worst = 0.0
    for s in range(0, d.shape[0], chunk):
        na = (a[s:s + chunk].double() ** 2).sum(1).numpy()
        ref = d_ref[s:s + chunk].astype(np.float64)
        tol = rtol * np.abs(ref) + atol_scale * (na[:, None] + nb[None, :])
        worst = max(worst, float((np.abs(d[s:s + chunk].astype(np.float64) - ref) / tol).max()))
    return worst


def oracle_subsample_parity(ev_factory, qf, gf, q_pids, g_pids, q_camids, g_camids, metric, sample_q):
    """Evaluate the first `sample_q` queries on one GPU and hold the result against the CPU side on the same inputs."""
    from oracle import restatement as R
    kind, ref = cpu_reference_path()
    sq = min(sample_q, qf.shape[0])
    ev = ev_factory()
    cmc, mAP, info = ev.evaluate(qf[:sq].cuda(), q_pids[:sq], q_camids[:sq], return_distmat=True)
    d = info["distmat"].cpu().numpy()
    d_ref = ref.compute_distance_matrix(qf[:sq], gf, metric).numpy()
    out = {"queries": sq, "cpu_side": kind}
    if metric == "euclidean":
        out["distance_max_err_over_tol"] = distance_ratio(d, d_ref, qf[:sq], gf)
        out["distance_tol"] = "1e-4*|d_ref| + 8e-7*(|q|^2+|g|^2)"
    else:
        out["distance_max_err_over_tol"] = float((np.abs(d - d_ref) / (1e-4 * np.abs(d_ref) + 2e-6)).max())
        out["distance_tol"] = "1e-4*|d_ref| + 2e-6"
    # ranking on IDENTICAL distances (ours): stable-argsort restatement of rank.py:103-171, and rank_cy where compiled
    cmc_o, map_o = R.evaluate_rank(d, q_pids[:sq], g_pids, q_camids[:sq], g_camids, max_rank=MAX_RANK)
    out["cmc_bit_exact"] = bool(np.array_equal(cmc, cmc_o))
    out["mAP_abs_err"] = abs(mAP - map_o)
    if kind == "reference" and R.count_row_ties(d) == 0:
        cmc_c, map_c = ref.evaluate_cy(d, q_pids[:sq], g_pids, q_camids[:sq], g_camids, MAX_RANK)
        out["rank_cy_cmc_bit_exact"] = bool(np.array_equal(cmc, cmc_c))
        out["rank_cy_mAP_abs_err"] = abs(mAP - float(map_c))          # rank_cy accumulates AP in float32
    out["num_ties"] = int(info["num_ties"])
    out["ok"] = bool(out["distance_max_err_over_tol"] <= 1.0 and out["cmc_bit_exact"] and out["mAP_abs_err"] < 1e-6)
    return out


# ------------------------------------------------------------------------------------------------------
# extras: the other BASELINE.json configs, one GPU
# ------------------------------------------------------------------------------------------------------
def cuda_time(fn, reps, flush=None):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = float("inf")
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def extra_c1_real_model(peaks):
    """Config C1: features of the reference's own (random-init) IEEE3modalPart, query set == gallery set."""
    from ieee_b200.engine import RetrievalEvaluator
    from oracle import restatement as R
    path = os.path.join(ROOT, "tests", "golden", "c1_real_model.npz")
    if not os.path.isfile(path):
        return {"skipped": "tests/golden/c1_real_model.npz missing"}
    g = np.load(path)
    f = torch.from_numpy(g["feats"])
    fd = f.cuda()
    Q = f.shape[0]

    def step():
        return RetrievalEvaluator(fd, g["pids"], g["camids"]).evaluate(fd, g["pids"], g["camids"], return_distmat=True)

    cmc, mAP, info = step()
    ms = cuda_time(step, 10)
    d = info["distmat"].cpu().numpy()
    truth = R.distance_fp64(f, f).numpy()
    cmc_t, map_t = R.evaluate_rank(truth.astype(np.float32), g["pids"], g["pids"], g["camids"], g["camids"])
    sec, kind, cores = time_cpu_path(f, f, g["pids"], g["pids"], g["camids"], g["camids"], "euclidean", 3, 1)
    return {"workload": f"real IEEE3modalPart features (random init, tests/golden/c1_real_model.npz) Q=G={Q} D={DIM} euclidean",
            "ms_per_step": ms, "queries_per_s": Q / (ms * 1e-3),
            "distance_max_err_over_tol_vs_reference": distance_ratio(d, g["distmat"], f, f),
            "max_abs_err_vs_fp64": {"ours": float(np.abs(d - truth).max()), "reference": float(np.abs(g["distmat"] - truth).max())},
            "mAP": mAP, "mAP_of_exact_distances": map_t, "mAP_reference_run": float(g["mAP"]),
            "cmc_equals_exact_ranking": bool(np.array_equal(cmc, cmc_t)),
            "cpu_baseline": {"value": Q / sec, "unit": "queries/s", "cores": cores, "kind": kind, "sample": "full C1 set, 3 passes"}}


def extra_cosine(ws, peaks):
    """Config C2 with the cosine metric (distance.py:67-80)."""
    from ieee_b200.engine import RetrievalEvaluator
    qf_d, gf_d = ws.qf.cuda(), ws.gf.cuda()
    lab = [torch.from_numpy(x).cuda() for x in (ws.q_pids, ws.q_camids, ws.g_pids, ws.g_camids)]
    Q = ws.qf.shape[0]

    def step():
        return RetrievalEvaluator(gf_d, lab[2], lab[3], "cosine", False, None, MAX_RANK).evaluate(qf_d, lab[0], lab[1])

    cmc, mAP, info = step()
    ms = cuda_time(step, 10)
    par = oracle_subsample_parity(lambda: RetrievalEvaluator(gf_d, lab[2], lab[3], "cosine", False, None, MAX_RANK), ws.qf, ws.gf,
                                  ws.q_pids, ws.g_pids, ws.q_camids, ws.g_camids, "cosine", REF_SAMPLE_Q)
    sq = REF_SAMPLE_Q
    sec, kind, cores = time_cpu_path(ws.qf[:sq], ws.gf, ws.q_pids[:sq], ws.g_pids, ws.q_camids[:sq], ws.g_camids, "cosine", 2, 1)
    return {"workload": f"market1501_shaped Q={Q} G={G_TOTAL} D={DIM} cosine max_rank={MAX_RANK}", "ms_per_step": ms,
            "queries_per_s": Q / (ms * 1e-3), "mAP": mAP, "rank1": float(cmc[0]), "parity": par,
            "cpu_baseline": {"value": sq / sec, "unit": "queries/s", "cores": cores, "kind": kind, "sample": cpu_sample_text(sq, cores)}}


def extra_rerank(peaks):
    """Config C3: k-reciprocal re-ranking (rerank.py:31, k1=20, k2=6, lambda=0.3) on an RGBNT201-shaped set."""
    from ieee_b200.metrics.distance import _device_distmat
    from ieee_b200.metrics.rank import evaluate_device
    from ieee_b200.testing import rgbnt201_shaped
    from ieee_b200.utils.rerank import re_ranking_device
    s = rgbnt201_shaped()
    qf, gf = s.qf.cuda(), s.gf.cuda()
    Q, G = qf.shape[0], gf.shape[0]
    N = Q + G
    qg, qq, gg = (_device_distmat(a, b, "euclidean") for a, b in ((qf, gf), (qf, qf), (gf, gf)))
    out = re_ranking_device(qg, qq, gg)
    ms_rr = cuda_time(lambda: re_ranking_device(qg, qq, gg), 10)

    def whole():
        a, b, c = (_device_distmat(x, y, "euclidean") for x, y in ((qf, gf), (qf, qf), (gf, gf)))
        d = re_ranking_device(a, b, c)
        return evaluate_device(d, s.q_pids, s.g_pids, s.q_camids, s.g_camids, MAX_RANK)

    ms_all = cuda_time(whole, 5)
    from oracle import restatement as R
    kind, ref = cpu_reference_path()
    mats = [m.cpu().numpy() for m in (qg, qq, gg)]
    t0 = time.perf_counter()
    ref_out = ref.re_ranking(mats[0], mats[1], mats[2], 20, 6, 0.3)
    cpu_s = time.perf_counter() - t0
    # query set == gallery set: every item meets its own copy at distance exactly 0, so the neighbour lists contain
    # exact ties.  rerank.py:48 leaves their order to NumPy's unstable argsort; ours (and the oracle restatement in its
    # stable mode) rank ties by index.  Parity is held against the stable restatement; the unmodified reference run is
    # reported beside it (it differs wherever its sort put a tie the other way round).
    stable_out = R.re_ranking(mats[0], mats[1], mats[2], 20, 6, 0.3, stable=True)
    ours = out.cpu().numpy()
    touched = 3 * 4 * N * N        # K1 reads the three raw blocks and writes the normalised N x N matrix, K2 reads it again
    return {"workload": f"rgbnt201_shaped Q=G={Q} (N={N}) k1=20 k2=6 lambda=0.3", "re_ranking_ms": ms_rr,
            "distances_rerank_evaluate_ms": ms_all, "touched_bytes": touched, "touched_gbs": touched / (ms_rr * 1e-3) / 1e9,
            "max_abs_err_vs_oracle_stable_ties": float(np.abs(ours - stable_out).max()), "tol": 1e-5,
            "ok": bool(np.abs(ours - stable_out).max() <= 1e-5),
            "max_abs_diff_vs_reference_unstable_argsort": float(np.abs(ours - ref_out).max()),
            "exact_ties_in_rows": int(R.count_row_ties(np.block([[mats[1], mats[0]], [mats[0].T, mats[2]]]))),
            "cpu_baseline": {"value": cpu_s * 1e3, "unit": "ms per re_ranking call", "cores": 1, "kind": kind,
                             "sample": "one call on the same three distance matrices (NumPy, single-threaded loops)"}}


def extra_c4_shard(peaks, check_q):
    """One gallery shard of config C4 as a single rank of an 8-way run sees it: 8192 queries x 125 000 gallery rows."""
    from ieee_b200.engine import PackedFeatures, RetrievalEvaluator, feature_center, packed_distmat
    from oracle import restatement as R
    dev = torch.device("cuda")
    Q, G, P, C = 8192, 125000, 12500, 8
    gen = torch.Generator(device=dev).manual_seed(4)
    centers = torch.randn(P + 1, DIM, device=dev, generator=gen)
    q_pids = torch.randint(1, P + 1, (Q,), device=dev, generator=gen)
    g_pids = torch.randint(1, P + 1, (G,), device=dev, generator=gen)
    q_cams = torch.randint(0, C, (Q,), device=dev, generator=gen)
    g_cams = torch.randint(0, C, (G,), device=dev, generator=gen)
    qf = torch.relu(centers[q_pids] + 2.75 * torch.randn(Q, DIM, device=dev, generator=gen))
    gf = torch.empty(G, DIM, device=dev)
    for s in range(0, G, 25000):
        gf[s:s + 25000] = torch.relu(centers[g_pids[s:s + 25000]] + 2.75 * torch.randn(25000, DIM, device=dev, generator=gen))
    del centers
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flops = 2.0 * Q * G * DIM
    pitch = (G + 31) // 32 * 32
    block = torch.empty((Q, pitch), dtype=torch.float32, device=dev)[:, :G]
    c = feature_center(qf)
    res = {"workload": f"C4-shaped shard: Q={Q} G={G} (1/8 of 1M) D={DIM} euclidean; synthetic, generated on the device (seed 4)"}
    for prec, centre in (("f16x3", c), ("bf16", None)):
        qp, gp = PackedFeatures(qf, "euclidean", False, prec, centre), PackedFeatures(gf, "euclidean", False, prec, centre)
        ms = cuda_time(lambda: packed_distmat(qp, gp, block), 3, flush)
        tf = flops / (ms * 1e-3) / 1e12
        res[f"gemm_{prec}"] = {"ms": ms, "tflops": tf, "frac_of_burst_peak": tf / peaks["bf16_tflops"],
                               "frac_of_sustained_peak": tf / peaks["bf16_tflops_sustained"]}
        del qp, gp
    del block

    def step(prec):
        ev = RetrievalEvaluator(gf, g_pids, g_cams, "euclidean", False, prec, MAX_RANK)
        return ev, ev.evaluate(qf, q_pids, q_cams)

    for prec in ("f16x3", "bf16"):
        ev, (cmc, mAP, info) = step(prec)
        ms = cuda_time(lambda: step(prec), 3)
        res[f"step_{prec}"] = {"ms": ms, "queries_per_s": Q / (ms * 1e-3), "mAP": mAP, "rank1": float(cmc[0]),
                               "equivalent_tflops": flops / (ms * 1e-3) / 1e12}
        del ev
    if check_q > 0:
        # SURVEY section 8(d): a query subsample against the CPU oracle over the full shard
        sq = min(check_q, Q)
        ev = RetrievalEvaluator(gf, g_pids, g_cams, "euclidean", False, "f16x3", MAX_RANK)
        cmc, mAP, info = ev.evaluate(qf[:sq], q_pids[:sq], q_cams[:sq], return_distmat=True)
        d = info["distmat"].cpu().numpy()
        qh, gh = qf[:sq].cpu(), gf.cpu()
        lab = [x.cpu().numpy() for x in (q_pids[:sq], g_pids, q_cams[:sq], g_cams)]
        kind, ref = cpu_reference_path()
        t0 = time.perf_counter()
        d_ref = ref.compute_distance_matrix(qh, gh, "euclidean").numpy()
        t1 = time.perf_counter()
        cmc_o, map_o = R.evaluate_rank(d, lab[0], lab[1], lab[2], lab[3], max_rank=MAX_RANK)
        t2 = time.perf_counter()
        res["parity"] = {"queries": sq, "cpu_side": kind, "distance_max_err_over_tol": distance_ratio(d, d_ref, qh, gh),
                         "distance_tol": "1e-4*|d_ref| + 8e-7*(|q|^2+|g|^2)", "cmc_bit_exact": bool(np.array_equal(cmc, cmc_o)),
                         "mAP_abs_err": abs(mAP - map_o), "num_ties": int(info["num_ties"])}
        res["parity"]["ok"] = bool(res["parity"]["distance_max_err_over_tol"] <= 1.0 and res["parity"]["cmc_bit_exact"]
                                   and res["parity"]["mAP_abs_err"] < 1e-6)
        cores = os.cpu_count() or 1
        res["cpu_baseline"] = {"value": sq / ((t1 - t0) + (t2 - t1)), "unit": "queries/s", "cores": cores, "kind": "port" if kind == "port" else "reference+port",
                               "sample": f"{sq} queries x the full {G}-row shard, one pass: torch CPU distance ({cores} threads, {t1 - t0:.1f} s) + "
                                         f"the oracle's NumPy ranking (stable argsort, {t2 - t1:.1f} s)"}
    return res


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def dump_outputs(path, cmc, mAP, info):
    """What the last timed step returned to its caller, one DIR/<name>.npy each (float32 CMC, the rest float64;
    counts and first-hit positions are exact in float64).  The workload is seeded, so two builds run with the same
    arguments can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    arrays = {"cmc": np.asarray(cmc, dtype=np.float32), "mAP": np.float64(mAP), "mINP": np.float64(info["mINP"]),
              "ap": info["ap"].cpu().numpy().astype(np.float64), "first": info["first"].cpu().numpy().astype(np.float64),
              "num_valid": np.float64(info["num_valid"]), "num_ties": np.float64(info["num_ties"])}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a))


def run_ours(args):
    import torch.distributed as dist
    from ieee_b200 import _lib
    from ieee_b200.engine import PackedFeatures, RetrievalEvaluator, feature_center, packed_distmat, shard_bounds
    from ieee_b200.metrics.rank import GalleryLabels, RankStages

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        print("bench.py: --gpus > 1 must be launched with torch.distributed.run; running on 1 GPU", file=sys.stderr)
    n_gpus = world
    _lib.require_cuda()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    lib = _lib.load()
    peaks = load_peaks()

    ws = make_workload(n_gpus)
    Q = ws.qf.shape[0]
    g0, g1 = shard_bounds(G_TOTAL, world, rank)
    gf_host = ws.gf[g0:g1].contiguous().pin_memory()
    qf_host = ws.qf.pin_memory()
    lab_host = [torch.from_numpy(x).pin_memory() for x in (ws.q_pids, ws.q_camids, ws.g_pids[g0:g1].copy(), ws.g_camids[g0:g1].copy())]

    def barrier():
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize()

    last_ev = [None]

    def step_device(qf, gf, qp, qc, gp, gc):
        ev = last_ev[0] = RetrievalEvaluator(gf, gp, gc, "euclidean", False, None, MAX_RANK, group=group, g_offset=g0, g_total=G_TOTAL)
        return ev.evaluate(qf, qp, qc)

    def step_e2e():
        # pinned host buffers in: labels and query features are copied first, the gallery features in row chunks on
        # a copy stream, each chunk packed and multiplied as it lands (RetrievalEvaluator.from_host)
        ev = RetrievalEvaluator.from_host(gf_host, lab_host[2], lab_host[3], "euclidean", False, None, MAX_RANK, group=group,
                                          g_offset=g0, g_total=G_TOTAL)
        return ev.evaluate(qf_host, lab_host[0], lab_host[1])

    def timed(fn, steps, warmup):
        # NVML is opened BEFORE the barrier: its first queries take 8 - 100 ms, and with that between the barrier and
        # rank 0's start event the other ranks' clocks were already running while they waited for rank 0's lists
        # (N = 2 read 1.29 ms per step instead of 0.88; N = 4 once 6.6 ms)
        sampler = ClockSampler(local_rank, enabled=rank == 0)      # rank 0 samples; the others stay quiet
        # as timeit does: no cyclic-GC pause inside the timed loop (a generation-2 collection of a process that has
        # imported torch takes milliseconds; with N ranks in lock step every rank waits for whoever collects).
        # Collected and switched off BEFORE the warm-up, for the same reason NVML is opened there.
        gc_was_on = gc.isenabled()
        gc.collect()
        gc.disable()
        sampler.arm()
        for _ in range(warmup):
            fn()
        barrier()
        at = {steps // 4, steps // 2, (3 * steps) // 4} if sampler.mode == "loop" else set()
        l0 = lib.ieee_launch_count()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        sampler.start()
        for i in range(steps):
            out = fn()
            if i in at:
                sampler.sample()
        stop.record()
        sampler.stop()
        if gc_was_on:
            gc.enable()
        launches = lib.ieee_launch_count() - l0
        if sampler.mode == "after":
            for i in range(steps):
                fn()
                if i in {steps // 4, steps // 2, (3 * steps) // 4}:
                    sampler.sample()
        barrier()
        clocks = sampler.result()
        ms = start.elapsed_time(stop)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
            ms = float(t.item())
        return ms, launches, clocks, out

    # ---- headline: inputs resident in HBM ------------------------------------------------------------
    qf_d, gf_d = qf_host.to(dev), gf_host.to(dev)
    lab_d = [t.to(dev) for t in lab_host]
    ms_dev, launches, clocks, out = timed(lambda: step_device(qf_d, gf_d, *lab_d), args.steps, args.warmup)
    cmc, mAP, info = out
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, cmc, mAP, info)
    value = Q * args.steps / (ms_dev / 1e3)
    count_path = ("fused into the contraction's epilogue (no distance block): %d of %d 128-output spans spilled for the exact recount"
                  % (last_ev[0].fused_stats["spilled_spans"], last_ev[0].fused_stats["spans"])) if info.get("fused") else (
        "staged: distance block written, gathered, counted (rank_count_warp_kernel)")

    # ---- end to end: pinned host buffers in, (cmc, mAP) on the host out ---------------------------------
    ms_e2e, _, _, _ = timed(step_e2e, args.steps, args.warmup)
    e2e_value = Q * args.steps / (ms_e2e / 1e3)
    # whole job: every rank copies its gallery shard and 1/N of the queries (all-gathered over NVLink) plus the labels
    h2d = (Q + G_TOTAL) * DIM * 4 + world * (2 * Q * 8) + 2 * G_TOTAL * 8
    d2h = 32 + 64 + 4 * MAX_RANK     # one result block per step: stats (32 B) + summary (64 B) + cmc

    # ---- per-kernel timing for the roofline (live, CUDA events on the launching stream) -------------------
    Gs = g1 - g0
    stage_ms = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    reps = max(3, min(args.steps, 10))

    def time_stage(name, fn):
        stage_ms[name] = cuda_time(fn, reps, flush)      # minimum: host hiccups between record() calls inflate the rest

    holder = {}
    centre = feature_center(qf_d)
    time_stage("feature_center", lambda: feature_center(qf_d))
    time_stage("pack_gallery", lambda: holder.__setitem__("g", PackedFeatures(gf_d, "euclidean", False, "f16x3", centre)))
    time_stage("pack_query", lambda: holder.__setitem__("q", PackedFeatures(qf_d, "euclidean", False, "f16x3", centre)))
    pitch = (Gs + 31) // 32 * 32          # the evaluator's scratch layout: 128-byte row pitch (TMA-store epilogue)
    dist_buf = torch.empty((Q, pitch), dtype=torch.float32, device=dev)[:, :Gs]
    time_stage("distmat_f16x3", lambda: packed_distmat(holder["q"], holder["g"], dist_buf))
    time_stage("group_gallery", lambda: holder.__setitem__("lab", GalleryLabels(lab_d[2], lab_d[3], dev)))
    gal = holder["lab"]
    cap = gal.list_cap(lab_d[0])
    st = RankStages(Q, cap, 1, dev)
    time_stage("rank_gather", lambda: st.gather(dist_buf, lab_d[0], lab_d[1], gal, g0))
    time_stage("rank_count", lambda: st.count(dist_buf, Gs, g0))
    time_stage("rank_finalize", lambda: st.finalize(G_TOTAL, MAX_RANK))
    g16 = PackedFeatures(gf_d, "euclidean", False, "bf16")
    q16 = PackedFeatures(qf_d, "euclidean", False, "bf16")
    time_stage("distmat_bf16_1pass", lambda: packed_distmat(q16, g16, dist_buf))
    del g16, q16, dist_buf, holder

    flops = 2.0 * Q * Gs * DIM
    gemm_tflops = flops / (stage_ms["distmat_f16x3"] * 1e-3) / 1e12
    gemm1_tflops = flops / (stage_ms["distmat_bf16_1pass"] * 1e-3) / 1e12
    count_gbs = 4.0 * Q * Gs / (stage_ms["rank_count"] * 1e-3) / 1e9
    traffic, traffic_1p, traffic_cnt = None, None, None
    tpath = next((p for p in (os.path.join(ROOT, "profiles", f) for f in ("r2_ncu_traffic.json", "r1_ncu_traffic.json")) if os.path.isfile(p)), None)
    if tpath is not None and n_gpus == 1:          # ncu capture of the same single-GPU shapes (bytes per launch)
        tj = json.load(open(tpath))
        rd = lambda k: tj[k]["dram_read_bytes"] + tj[k]["dram_write_bytes"] if k in tj else None
        traffic, traffic_1p, traffic_cnt = rd("distmat_umma_chunked_kernel"), rd("distmat_umma_kernel_bf16_1pass"), rd("rank_count_warp_kernel")
    chunk = lib.ieee_set_accum_chunk(-1)
    roofline = {"kernel": "distmat_umma_chunked_kernel<2> (cta_group::2; f16x3: fp16 hi/lo split of the centred operands, 3 tcgen05 "
                          f"passes per k block, cross terms first, accumulation chunked every {chunk} K-slices)",
                "bound": "tensor", "achieved": gemm_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": gemm_tflops / peaks["bf16_tflops"], "traffic": traffic,
                "peak_source": peaks["source"] + " (burst: the kernel is timed alone)",
                "issued_tflops": 3 * gemm_tflops, "issued_frac": 3 * gemm_tflops / peaks["bf16_tflops"],
                "algorithmic_flops_per_launch": flops,
                "note": "achieved counts ALGORITHMIC flops 2*Q*G*D once; the fp32-grade split issues 3x that on the tensor "
                        f"pipe (issued_*). traffic = DRAM bytes per launch from {os.path.basename(tpath) if tpath else 'n/a'}"}
    extra = {
        "roofline_bf16_1pass": {"kernel": "distmat_umma_kernel<2> (cta_group::2; one tcgen05 pass on bf16-rounded features; not parity grade "
                                          "for f32 inputs, exact for bf16 inputs)", "bound": "tensor", "achieved": gemm1_tflops,
                                "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": gemm1_tflops / peaks["bf16_tflops"],
                                "traffic": traffic_1p},
        "roofline_rank_count": {"kernel": f"rank_count_warp_kernel<1> (one warp per query; {Q} rows of {Gs} columns)", "bound": "hbm",
                                "achieved": count_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": count_gbs / peaks["hbm_gbs"],
                                "algorithmic_bytes": 4 * Q * Gs, "traffic": traffic_cnt},
        "stage_ms": {k: round(v, 4) for k, v in stage_ms.items()},
    }

    # ---- parity, in the record: sharded == single GPU, and a query subsample against the CPU side --------------
    parity = None
    if rank == 0 and not args.no_parity:
        gf_full = ws.gf.to(dev) if world > 1 else gf_d
        make_ev = lambda: RetrievalEvaluator(gf_full, ws.g_pids, ws.g_camids, "euclidean", False, None, MAX_RANK)
        parity = {}
        if world > 1:
            c1, m1, i1 = make_ev().evaluate(qf_d, ws.q_pids, ws.q_camids)
            parity["sharded_equals_single_gpu"] = bool(np.array_equal(c1, cmc) and m1 == mAP and torch.equal(i1["ap"], info["ap"])
                                                       and torch.equal(i1["first"], info["first"]) and i1["num_ties"] == info["num_ties"])
            parity["single_gpu_mAP"] = m1
        parity["oracle_subsample"] = oracle_subsample_parity(make_ev, ws.qf, ws.gf, ws.q_pids, ws.g_pids, ws.q_camids, ws.g_camids,
                                                             "euclidean", REF_SAMPLE_Q)
        parity["ok"] = bool(parity["oracle_subsample"]["ok"] and parity.get("sharded_equals_single_gpu", True))
        del gf_full

    line = None
    if rank == 0:
        cpu_baseline = None
        if n_gpus == 1 and not args.no_cpu_baseline:
            sec, kind, cores = time_cpu_path(ws.qf, ws.gf, ws.q_pids, ws.g_pids, ws.q_camids, ws.g_camids, "euclidean", 2, 1)
            cpu_baseline = {"value": Q_BASE / sec, "unit": "queries/s", "cores": cores, "kind": kind,
                            "sample": f"full workload ({Q_BASE} x {G_TOTAL}), 1 warm-up + 2 timed passes; torch CPU distance "
                                      f"({cores} threads) + rank_cy.evaluate_cy (single-threaded by construction)",
                            "ms_per_step": 1e3 * sec}
        if n_gpus == 1 and not args.no_extras:
            del qf_d, gf_d
            torch.cuda.empty_cache()
            extra["extras"] = {}
            for name, fn in (("c1_real_model", lambda: extra_c1_real_model(peaks)), ("c2_cosine", lambda: extra_cosine(ws, peaks)),
                             ("c3_rerank", lambda: extra_rerank(peaks)), ("c4_shard", lambda: extra_c4_shard(peaks, args.c4_check))):
                try:
                    extra["extras"][name] = fn()
                except Exception as e:          # an extra must never cost the headline
                    extra["extras"][name] = {"error": repr(e)[:300]}
                torch.cuda.empty_cache()
        line = {
            "metric": METRIC_NAME, "value": value, "unit": "queries/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16x3 split of f32 (fp32-equivalent products, f32 accumulate); rank: u32/i32; AP: f64",
            "data": "synthetic", "config": bench_config(n_gpus),
            "count_path": count_path,
            "exchange": ("none (one GPU)" if world == 1 else os.environ.get("IEEE_B200_EXCHANGE", "peer") +
                         (": stores into NVLink peer memory from the rank kernels, flag hand-over, no collective launches per step"
                          if os.environ.get("IEEE_B200_EXCHANGE", "peer") == "peer" else ": all-gather + all-reduce launches")),
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "result": {"mAP": mAP, "rank1": float(cmc[0]), "mINP": info.get("mINP"), "num_valid": int(info["num_valid"]),
                       "num_ties": int(info["num_ties"]), "parity": parity},
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier(group=group)
        dist.destroy_process_group()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--c4-check", type=int, default=2048, help="query subsample of the C4-shaped shard held against the CPU oracle (0: off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline step's results of the last timed step to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
