"""Dense ieee_rerank of another build of the library (e.g. the commit before the streamed form was added) against this
tree's build, on seeded inputs: the outputs must be bit-identical.

    git worktree add /tmp/parent <commit> && (cd /tmp/parent && python -m ieee_b200.build)
    python profiles/rerank_dense_compare.py --other-lib /tmp/parent/ieee_b200/libieee_b200.so [--out FILE]
"""
import argparse
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ieee_b200 import _lib                                                                      # noqa: E402
from ieee_b200.metrics.distance import _device_distmat                                          # noqa: E402
from ieee_b200.testing import make_retrieval_set, market1501_shaped, rgbnt201_shaped            # noqa: E402


def run(lib, qg, qq, gg, k1, k2, lam):
    Q, G = qg.shape
    out = torch.full((Q, G), float("nan"), device="cuda")
    nbytes = lib.ieee_rerank_workspace_bytes(Q, G, k1, k2)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    rc = lib.ieee_rerank(qg.data_ptr(), qg.stride(0), qq.data_ptr(), qq.stride(0), gg.data_ptr(), gg.stride(0), Q, G, k1, k2,
                         lam, out.data_ptr(), out.stride(0), ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.ieee_last_error()
    torch.cuda.synchronize()
    return out, nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other-lib", required=True)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    this = _lib.load()
    other = C.CDLL(os.path.abspath(a.other_lib))
    for n in ("ieee_rerank", "ieee_rerank_workspace_bytes", "ieee_last_error"):
        getattr(other, n).restype, getattr(other, n).argtypes = _lib.SIGNATURES[n]
    sets = [("rgbnt201", rgbnt201_shaped()), ("market", market1501_shaped())]
    sets += [("r%d" % i, make_retrieval_set(q, g, 20, 4, dim=d, sigma=2.0, seed=i))
             for i, (q, g, d) in enumerate([(37, 150, 96), (1000, 5003, 320), (5, 16, 48), (420, 1900, 256)])]
    lines, bad = [], 0
    for name, s in sets:
        qf, gf = s.qf.cuda(), s.gf.cuda()
        mats = [_device_distmat(x, y, "euclidean") for x, y in ((qf, gf), (qf, qf), (gf, gf))]
        N = qf.shape[0] + gf.shape[0]
        for k1, k2, lam in ((20, 6, 0.3), (20, 1, 0.3), (30, 8, 0.3), (10, 4, 0.0)):
            if k1 + 1 > N:
                continue
            x, bx = run(other, *mats, k1, k2, lam)
            y, by = run(this, *mats, k1, k2, lam)
            same = torch.equal(x, y) and bx == by
            bad += not same
            lines.append("%-9s Q=%5d G=%5d k1=%2d k2=%d lambda=%.1f  identical=%s  (workspace %d / %d bytes)"
                         % (name, qf.shape[0], gf.shape[0], k1, k2, lam, same, bx, by))
    lines.append("dense ieee_rerank, other build vs this build: " + ("all identical" if bad == 0 else "%d differ" % bad))
    text = "\n".join(lines) + "\n"
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)
    print(text)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
