"""Dense GNN re-ranking (gnn_reranking_distmat: ieee_gnn_rerank + both contractions) and dense k-reciprocal re-ranking
(ieee_rerank) of another build of the library (e.g. the commit before the streamed GNN form was added) against this
tree's build, on seeded inputs: the outputs must be bit-identical.

    git worktree add /tmp/parent <commit> && (cd /tmp/parent && python -m ieee_b200.build)
    python profiles/gnn_dense_compare.py --other-lib /tmp/parent/ieee_b200/libieee_b200.so [--out FILE]
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
from ieee_b200.utils.gnn_reranking import gnn_reranking_distmat                                  # noqa: E402
from ieee_b200.utils.rerank import re_ranking_device                                             # noqa: E402


def with_lib(lib, fn):
    """Run fn with `lib` as the library every ieee_b200 call goes through."""
    saved = _lib._lib
    _lib._lib = lib
    try:
        out = fn()
        torch.cuda.synchronize()
        return out
    finally:
        _lib._lib = saved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other-lib", required=True)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    this = _lib.load()
    other = C.CDLL(os.path.abspath(a.other_lib))
    for n, (res, args) in _lib.SIGNATURES.items():
        if hasattr(other, n):
            getattr(other, n).restype, getattr(other, n).argtypes = res, args
    sets = [("c3", rgbnt201_shaped()), ("market", market1501_shaped())]
    sets += [("r%d" % i, make_retrieval_set(q, g, 20, 4, dim=d, sigma=2.0, seed=i))
             for i, (q, g, d) in enumerate([(37, 150, 96), (5, 16, 48), (420, 1900, 256)])]
    lines, bad = [], 0
    for name, s in sets:
        qf, gf = s.qf.cuda(), s.gf.cuda()
        xq, xg = (torch.nn.functional.normalize(x, dim=1) for x in (qf, gf))
        N = qf.shape[0] + gf.shape[0]
        for k1, k2 in ((26, 7), (20, 6), (10, 1)):
            if k1 > N:
                continue
            x = with_lib(other, lambda: gnn_reranking_distmat(xq, xg, k1, k2))
            y = with_lib(this, lambda: gnn_reranking_distmat(xq, xg, k1, k2))
            same = torch.equal(x, y)
            bad += not same
            lines.append("%-7s Q=%5d G=%5d gnn          k1=%2d k2=%d  identical=%s" % (name, qf.shape[0], gf.shape[0], k1, k2, same))
        mats = [_device_distmat(p, q, "euclidean") for p, q in ((qf, gf), (qf, qf), (gf, gf))]
        if 21 <= N:
            x = with_lib(other, lambda: re_ranking_device(*mats))
            y = with_lib(this, lambda: re_ranking_device(*mats))
            same = torch.equal(x, y)
            bad += not same
            lines.append("%-7s Q=%5d G=%5d k-reciprocal k1=20 k2=6  identical=%s" % (name, qf.shape[0], gf.shape[0], same))
    lines.append("dense re-ranking, other build vs this build: " + ("all identical" if bad == 0 else "%d differ" % bad))
    text = "\n".join(lines) + "\n"
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)
    print(text)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
