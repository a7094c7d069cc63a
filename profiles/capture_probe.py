"""evaluate() against the replay of a captured step (RetrievalEvaluator.capture) at the Market shape (3368 x 15913 x
2304, f16x3), on one GPU and -- when the box has two -- over a gallery sharded across two GPUs (peer exchange).

Both forms are warmed up, then alternated call by call for --steps steps each.  Per call: a CUDA event on the current
stream before it and one after it returns (both calls end with the result on the host, so the interval is the step as
a caller sees it, host share included), and the host clock around it.  Medians and 10th / 90th percentiles, plus
whether the replay's cmc, mAP, mINP, ap and first equal evaluate()'s.  The labels are device tensors, so evaluate()
takes its steady-state route (capacity memo hit: one foreign call).

    python profiles/capture_probe.py [--steps 300] [--out FILE]
"""
import argparse
import os
import socket
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ieee_b200.engine import RetrievalEvaluator, shard_bounds     # noqa: E402
from ieee_b200.testing import market1501_shaped                    # noqa: E402


def timed(fn, steps_out):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    out = fn()
    t1 = time.perf_counter()
    e1.record()
    e1.synchronize()
    steps_out.append((e0.elapsed_time(e1), (t1 - t0) * 1e3))
    return out


def stats(rows):
    a = np.array(rows)
    return "  ".join("%s median %.3f ms (p10 %.3f, p90 %.3f)" % (what, np.median(a[:, i]), np.percentile(a[:, i], 10),
                                                                 np.percentile(a[:, i], 90))
                     for i, what in enumerate(("events", "host clock")))


def measure(ev, qf, qp, qc, steps, warmup=30):
    h = ev.capture(qf, qp, qc)
    for _ in range(warmup):
        ev.evaluate(qf, qp, qc)
        h.replay()
    a, b = ev.evaluate(qf, qp, qc), h.replay()
    same = (np.array_equal(a[0], b[0]) and a[1] == b[1] and a[2]["mINP"] == b[2]["mINP"]
            and torch.equal(a[2]["ap"], b[2]["ap"]) and torch.equal(a[2]["first"], b[2]["first"]))
    ev_t, rp_t = [], []
    for _ in range(steps):
        timed(lambda: ev.evaluate(qf, qp, qc), ev_t)
        timed(h.replay, rp_t)
    return ("evaluate()  %s\nreplay()    %s\nreplay equals evaluate bit for bit: %s"
            % (stats(ev_t), stats(rp_t), "yes" if same else "NO"))


def labels(s, dev, g0, g1):
    t = lambda x: torch.from_numpy(x).to(dev)         # noqa: E731
    return t(s.q_pids), t(s.q_camids), t(s.g_pids[g0:g1]), t(s.g_camids[g0:g1])


def two_gpu_worker(rank, world, port, steps, out_path):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    s = market1501_shaped()
    G = s.gf.shape[0]
    g0, g1 = shard_bounds(G, world, rank)
    qp, qc, gp, gc = labels(s, dev, g0, g1)
    ev = RetrievalEvaluator(s.gf[g0:g1].to(dev), gp, gc, group=dist.group.WORLD, g_offset=g0, g_total=G)
    text = measure(ev, s.qf.to(dev), qp, qc, steps)
    if rank == 0:
        with open(out_path, "w") as f:
            f.write(text)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    n_gpu = torch.cuda.device_count()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# capture_probe, 3368 x 15913 x 2304 f16x3, %d steps of each form after warm-up, on %s (name, power limit, "
             "max SM clock); %d GPU(s) in the box" % (a.steps, gpu[0] if gpu else "?", n_gpu), ""]
    dev = torch.device("cuda", 0)
    s = market1501_shaped()
    qp, qc, gp, gc = labels(s, dev, 0, s.gf.shape[0])
    ev = RetrievalEvaluator(s.gf.to(dev), gp, gc)
    lines += ["## one GPU", measure(ev, s.qf.to(dev), qp, qc, a.steps), ""]
    del ev
    lines.append("## gallery sharded across two GPUs (peer exchange), rank 0")
    if n_gpu >= 2:
        import torch.multiprocessing as mp
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        with tempfile.TemporaryDirectory() as tmp:
            out_path = os.path.join(tmp, "two.txt")
            mp.spawn(two_gpu_worker, args=(2, port, a.steps, out_path), nprocs=2, join=True)
            lines.append(open(out_path).read())
    else:
        lines.append("not measured (the box has %d GPU)" % n_gpu)
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
