"""GPU parity: distance matrix through the drop-in API / C ABI vs the CPU oracle (same seeded inputs)."""
import os

import numpy as np
import pytest
import torch

from oracle import restatement as R
from ieee_b200 import _lib
from ieee_b200.metrics import compute_distance_matrix
from ieee_b200.metrics.distance import _device_distmat
from ieee_b200.testing import make_retrieval_set, rgbnt201_shaped

pytestmark = pytest.mark.gpu

RTOL = 1e-4          # north_star: distances within 1e-4 relative in fp32
CANCEL_ULPS = 4e-7   # a few fp32 ulps of |q|^2 + |g|^2: the cancellation floor the reference itself sits on (F7)
# The tcgen05 fp32 accumulator truncates instead of rounding (profiles/accuracy_r2.txt).  The F16X3 path therefore
# (a) packs euclidean operands relative to the query set's mean, which removes the one-signed drift on post-ReLU
# features and shrinks the cancellation scale, (b) closes the TMEM accumulator every 4 K-slices and sums the chunks in
# fp32 registers (round to nearest), and (c) issues the small cross terms of a chunk before its hi*hi products, so only
# 16 truncations per chunk happen at full magnitude.  What is left is no more than the reference's own floor.
TC_ACCUM_FLOOR = 4e-7            # F16X3, default chunking (both cta_group modes), in units of |q|^2 + |g|^2
TC_ACCUM_FLOOR_UNCHUNKED = 2e-5  # whole-K accumulation in TMEM (BF16 1-pass mode, ieee_set_accum_chunk(0))
SPLIT_EPS = 2.0 ** -21   # fp16 hi+lo keeps 22 mantissa bits per operand: each product is off by <= ~2^-21 relative


def parity_terms(a, b, metric):
    """What assert_distance_parity measures against: (fp64 truth, the reference's fp32 result, |q|^2+|g|^2,
    sqrt(sum_k (a_k b_k)^2)).  Worth computing once when several results of the same inputs are checked."""
    truth = R.distance_fp64(a, b, metric).numpy()
    ref = R.compute_distance_matrix(a, b, metric).numpy()
    a64, b64 = a.double(), b.double()
    if metric == "cosine":
        a64 = a64 / a64.norm(dim=1, keepdim=True).clamp_min(1e-12)
        b64 = b64 / b64.norm(dim=1, keepdim=True).clamp_min(1e-12)
    scale = ((a64 ** 2).sum(1, keepdim=True) + (b64 ** 2).sum(1, keepdim=True).t()).numpy()
    prod_rms = torch.sqrt((a64 ** 2) @ (b64 ** 2).t()).numpy()
    return truth, ref, scale, prod_rms


def assert_distance_parity(got, a, b, metric, rtol=RTOL, split=True, floor=None, terms=None):
    """|got - fp64 truth| <= rtol*|truth| + floor.

    floor = the cancellation floor the reference's own fp32 GEMM sits on (a few ulps of |q|^2+|g|^2) plus, for
    the f16x3 split, 4 sigma of its rounding model: independent per-product errors of 2^-21 relative, i.e.
    2 * 4 * 2^-21 * sqrt(sum_k (a_k b_k)^2)  (~ 1e-8 relative at D=2304: below the fp32 floor).
    `terms`: parity_terms(a, b, metric), when the caller already has them.
    """
    truth, ref, scale, prod_rms = terms if terms is not None else parity_terms(a, b, metric)
    alpha = 2.0 if metric == "euclidean" else 1.0
    tol = rtol * np.abs(truth) + CANCEL_ULPS * scale
    if split:   # tensor-core path
        unchunked = _lib.load().ieee_set_accum_chunk(-1) == 0   # (negative: query only)
        tol = tol + alpha * 4 * SPLIT_EPS * prod_rms + (floor or (TC_ACCUM_FLOOR_UNCHUNKED if unchunked else TC_ACCUM_FLOOR)) * scale
    err = np.abs(got.astype(np.float64) - truth)
    assert (err <= tol).all(), f"max err/tol = {(err / tol).max():.3g}"
    ref_err = np.abs(ref.astype(np.float64) - truth)
    return float((err / np.maximum(np.abs(truth), 1e-30)).max()), float(err.max()), float(ref_err.max())


def features(q, g, d, seed=0):
    gen = torch.Generator().manual_seed(seed)
    return torch.relu(torch.randn(q, d, generator=gen) + 0.3), torch.relu(torch.randn(g, d, generator=gen) + 0.3)


@pytest.fixture(params=[1, 2], ids=["cta_group1", "cta_group2"])
def cta_group(request):
    prev = _lib.load().ieee_set_cta_group(request.param)
    yield request.param
    _lib.load().ieee_set_cta_group(prev)


SHAPES = [(10, 100, 2048), (1, 1, 64), (130, 300, 96), (257, 513, 2304), (128, 256, 64), (300, 1000, 200), (5, 7, 3)]


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_f16x3_matches_oracle(cta_group, shape, metric):
    a, b = features(*shape, seed=sum(shape))
    out = compute_distance_matrix(a.cuda(), b.cuda(), metric)
    assert out.is_cuda and out.dtype == torch.float32 and tuple(out.shape) == shape[:2]
    assert_distance_parity(out.cpu().numpy(), a, b, metric)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_golden_distance(golden_dir, metric):
    g = np.load(os.path.join(golden_dir, "distance_small.npz"))
    a, b = torch.from_numpy(g["a"]), torch.from_numpy(g["b"])
    out = compute_distance_matrix(a, b, metric)        # CPU tensors in -> CPU tensor out, like the reference
    assert not out.is_cuda and out.dtype == torch.float32
    np.testing.assert_allclose(out.numpy(), g[metric], rtol=1e-4, atol=1e-4 if metric == "euclidean" else 1e-6)
    if metric == "cosine":
        assert (out.numpy()[:, 3] == 1.0).all()        # all-zero row -> exactly 1 (distance.py:77-79)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_fp32_simt_matches_oracle(metric):
    a, b = features(70, 130, 300, seed=5)
    out = compute_distance_matrix(a.cuda(), b.cuda(), metric, precision="fp32_simt")
    assert_distance_parity(out.cpu().numpy(), a, b, metric, split=False)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_bf16_single_pass_is_exact_for_bf16_inputs(cta_group, metric):
    a, b = features(200, 700, 512, seed=9)
    a16, b16 = a.bfloat16(), b.bfloat16()
    out = compute_distance_matrix(a16.cuda(), b16.cuda(), metric)
    assert out.dtype == torch.bfloat16                     # output dtype follows the inputs (distance.py)
    got = _device_distmat(a16.cuda(), b16.cuda(), metric).cpu().numpy()
    if metric == "euclidean":                              # products of bf16 values are exact in fp32
        assert_distance_parity(got, a16.float(), b16.float(), metric, floor=TC_ACCUM_FLOOR_UNCHUNKED)
    else:                                                  # normalised rows are re-rounded to bf16: bf16-level accuracy
        truth = R.distance_fp64(a16.float(), b16.float(), metric).numpy()
        assert np.abs(got - truth).max() < 1e-2


def test_tensor_path_agrees_with_simt_path(cta_group):
    s = make_retrieval_set(300, 700, 30, 4, dim=2304, seed=2)
    x3 = compute_distance_matrix(s.qf.cuda(), s.gf.cuda(), "euclidean").cpu().numpy()
    simt = compute_distance_matrix(s.qf.cuda(), s.gf.cuda(), "euclidean", precision="fp32_simt").cpu().numpy()
    assert np.abs(x3 - simt).max() <= 1e-4 * np.abs(simt).max()


def test_normalize_feature_then_euclidean():
    """engine.py:391-394 then distance.py:59-64."""
    a, b = features(64, 200, 2304, seed=3)
    an, bn = torch.nn.functional.normalize(a, p=2, dim=1), torch.nn.functional.normalize(b, p=2, dim=1)
    got = _device_distmat(a.cuda(), b.cuda(), "euclidean", normalize=True).cpu().numpy()
    assert_distance_parity(got, an, bn, "euclidean")


def test_full_dim_relative_error_is_within_1e4():
    """At the path's real feature width (D = 2304) the f16x3 result is within 1e-4 RELATIVE of the fp64
    distance for every pair that is not a near-duplicate (d > 1e-3 (|q|^2+|g|^2)); no floor needed."""
    s = make_retrieval_set(400, 1500, 30, 4, dim=2304, seed=7)
    out = compute_distance_matrix(s.qf.cuda(), s.gf.cuda()).cpu().numpy().astype(np.float64)
    truth = R.distance_fp64(s.qf, s.gf).numpy()
    ref = R.compute_distance_matrix(s.qf, s.gf).numpy().astype(np.float64)
    scale = ((s.qf.double() ** 2).sum(1, keepdim=True) + (s.gf.double() ** 2).sum(1, keepdim=True).t()).numpy()
    mask = truth > 1e-3 * scale
    rel = (np.abs(out - truth) / np.abs(truth))[mask].max()
    rel_ref = (np.abs(ref - truth) / np.abs(truth))[mask].max()
    print(f"max relative error vs fp64: ours {rel:.3e}, reference fp32 {rel_ref:.3e}")
    assert rel < 1e-4 and mask.mean() > 0.99
    assert (np.abs(out - ref) <= 1e-4 * np.abs(ref))[mask].all()      # and within 1e-4 of the reference itself


def test_rgbnt201_shape_self_distances():
    s = rgbnt201_shaped()
    out = compute_distance_matrix(s.qf.cuda(), s.gf.cuda()).cpu().numpy()
    rel, abs_err, ref_abs = assert_distance_parity(out, s.qf, s.gf, "euclidean")
    diag = np.abs(np.diag(out))
    assert diag.max() < TC_ACCUM_FLOOR * 2 * (s.qf ** 2).sum(1).max().item()    # squared, unclamped, ~0 (F7)


def test_accumulation_chunking_improves_accuracy():
    """ieee_set_accum_chunk: whole-K accumulation in TMEM vs chunks of 4 and 1 K-slices; centring switched off so
    that the non-negative features make the truncation a one-signed drift (the case chunking exists for)."""
    s = make_retrieval_set(256, 700, 20, 4, dim=2304, seed=3)
    truth = R.distance_fp64(s.qf, s.gf).numpy()
    scale = ((s.qf.double() ** 2).sum(1, keepdim=True) + (s.gf.double() ** 2).sum(1, keepdim=True).t()).numpy()
    lib, errs = _lib.load(), {}
    prev, prev_c = lib.ieee_set_accum_chunk(4), lib.ieee_set_centering(0)
    try:
        for chunk in (0, 4, 1):
            lib.ieee_set_accum_chunk(chunk)
            out = compute_distance_matrix(s.qf.cuda(), s.gf.cuda()).cpu().numpy().astype(np.float64)
            errs[chunk] = float((np.abs(out - truth) / scale).max())
    finally:
        lib.ieee_set_accum_chunk(prev)
        lib.ieee_set_centering(prev_c)
    assert errs[0] < TC_ACCUM_FLOOR_UNCHUNKED and errs[4] < 1e-6 and errs[1] <= 1.2 * errs[4] and errs[4] < errs[0] / 3, errs


def test_centering_removes_the_cancellation_scale(golden_dir):
    """Real-model features (post-ReLU, |x|^2 ~ 1.6e5, distances ~ 1e2): relative to the query mean the same pairs
    have |x'|^2 ~ 6e1, and the error drops from ~1e-7 (|q|^2 + |g|^2) to far below the reference's own."""
    g = np.load(os.path.join(golden_dir, "c1_real_model.npz"))
    f = torch.from_numpy(g["feats"])
    truth = R.distance_fp64(f, f).numpy()
    ref_err = np.abs(g["distmat"].astype(np.float64) - truth).max()
    lib = _lib.load()
    errs = {}
    prev, prev_dbg = lib.ieee_set_centering(-1), lib.ieee_set_debug_flags(0)
    try:
        for on in (0, 1):
            lib.ieee_set_centering(on)
            for prec in ("f16x3", "fp32_simt"):
                out = compute_distance_matrix(f.cuda(), f.cuda(), precision=prec).cpu().numpy().astype(np.float64)
                errs[(on, prec)] = float(np.abs(out - truth).max())
        # without the centre EVERY pair of this set is a near duplicate (d ~ 1e2 against a scale of 3e5): the fix-up pass
        # recomputes them all; switched off as well (debug bit 5), the accumulator's floor shows
        lib.ieee_set_centering(0)
        lib.ieee_set_debug_flags(32)
        out = compute_distance_matrix(f.cuda(), f.cuda()).cpu().numpy().astype(np.float64)
        errs["expansion only"] = float(np.abs(out - truth).max())
    finally:
        lib.ieee_set_centering(prev)
        lib.ieee_set_debug_flags(prev_dbg)
    print("max |d - fp64| on c1_real_model: reference %.3g; ours %s" % (ref_err, errs))
    assert errs[(1, "f16x3")] < 0.05 * ref_err and errs[(1, "fp32_simt")] < 0.05 * ref_err
    assert errs[(0, "f16x3")] < 0.05 * ref_err                       # fix-up alone
    assert errs[(1, "f16x3")] < 0.01 * errs["expansion only"] and errs["expansion only"] > 0.5 * ref_err


def test_feature_center_is_the_sample_mean():
    from ieee_b200.engine import feature_center
    gen = torch.Generator().manual_seed(4)
    for rows, D in ((1000, 2304), (37, 100), (1, 5), (5000, 515)):
        x = torch.relu(torch.randn(rows, D, generator=gen) + 0.3)
        n_s = min(rows, 64)
        sample = x[:: rows // n_s][:n_s]
        c = feature_center(x.cuda()).cpu()
        torch.testing.assert_close(c, sample.mean(0), rtol=1e-5, atol=1e-6)
        cn = feature_center(x.cuda(), normalize=True).cpu()
        m = sample.mean(0)
        torch.testing.assert_close(cn, m / m.norm().clamp_min(1e-12), rtol=1e-5, atol=1e-6)
        assert torch.equal(c, feature_center(x.cuda()).cpu())          # deterministic


def test_same_centre_for_both_operands_is_enforced():
    from ieee_b200.engine import PackedFeatures, feature_center, packed_distmat
    a, b = features(40, 90, 128, seed=8)
    c = feature_center(a.cuda())
    qa, gb = PackedFeatures(a.cuda(), "euclidean", False, "f16x3", c), PackedFeatures(b.cuda(), "euclidean", False, "f16x3", c)
    out = torch.empty(40, 96, device="cuda")[:, :90]
    packed_distmat(qa, gb, out)
    assert_distance_parity(out.cpu().numpy(), a, b, "euclidean")
    with pytest.raises(AssertionError):
        packed_distmat(qa, PackedFeatures(b.cuda(), "euclidean", False, "f16x3"), out)
    with pytest.raises(_lib.IeeeB200Error):                        # cosine is not translation invariant
        PackedFeatures(a.cuda(), "cosine", False, "f16x3", c)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_second_device_in_one_process():
    """Kernel attributes (dynamic shared memory) are per device: evaluate on cuda:0, then on cuda:1."""
    a, b = features(300, 600, 2304, seed=12)
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        outs.append(compute_distance_matrix(a.to(dev), b.to(dev)).cpu().numpy())
        assert_distance_parity(outs[-1], a, b, "euclidean")
    assert np.array_equal(outs[0], outs[1])


def test_argument_errors():
    a, b = features(4, 5, 8)
    with pytest.raises(ValueError):
        compute_distance_matrix(a.cuda(), b.cuda(), "manhattan")
    with pytest.raises(AssertionError):
        compute_distance_matrix(a.cuda(), b.cuda()[:, :4])
    with pytest.raises(AssertionError):
        compute_distance_matrix(a.cuda()[0], b.cuda())
    assert compute_distance_matrix(a.cuda()[:0], b.cuda()).shape == (0, 5)


def test_noncontiguous_rows_and_views():
    a, b = features(40, 90, 128, seed=8)
    big = torch.zeros(40, 256).cuda()
    big[:, :128] = a.cuda()
    out = compute_distance_matrix(big[:, :128], b.cuda())        # row stride 256, unit column stride
    assert_distance_parity(out.cpu().numpy(), a, b, "euclidean")
