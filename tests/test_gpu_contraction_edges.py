"""GPU parity of the contraction where its simple paths end: near-duplicate fix-ups past the list's capacity, CTAs that
loop over many tiles with ragged edges, every accumulation chunking, raster panel and store epilogue, and the whole-K
kernel -- each against a float64 reference of the same inputs."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import restatement as R
from ieee_b200 import _lib, engine
from ieee_b200.engine import PackedFeatures, RetrievalEvaluator, feature_center, packed_distmat
from ieee_b200.metrics import compute_distance_matrix
from ieee_b200.metrics.distance import _device_distmat
from test_gpu_distance import (CANCEL_ULPS, RTOL, TC_ACCUM_FLOOR, TC_ACCUM_FLOOR_UNCHUNKED, assert_distance_parity,
                               cta_group, features, parity_terms)  # noqa: F401  (cta_group is a fixture)

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def knob(setter, value):
    """Set one of the library's process-global ieee_set_* knobs for the duration of a block."""
    prev = setter(value)
    try:
        yield
    finally:
        setter(prev)


def accum_chunk(chunk):
    """ieee_set_accum_chunk(chunk) for a block; None keeps the default."""
    return contextlib.nullcontext() if chunk is None else knob(_lib.load().ieee_set_accum_chunk, chunk)


# ---------------------------------------------------------------------------------------------------------------------
# Near-duplicate fix-ups past the list's capacity
# ---------------------------------------------------------------------------------------------------------------------
# 512 base rows, each copied 32 times to gallery positions b + 512 j: every copy sits in a different 128-column span, so
# every query row flags 32 spans -- 16 384 in all, against a list of 2 Q + 4096 = 5120 entries.
NB, NCOPY, DIM = 512, 32, 2304
NEAR_EPS = 0.02      # copies relu(base + eps * noise): d ~ 3e-4 .. 4e-4 of the centred |q'|^2 + |g'|^2
NEAR_BOUND = 1e-5    # relative to d: the difference form holds ~1e-7 d; the expansion alone misses it by far


def scattered_copies(eps, seed):
    gen = torch.Generator().manual_seed(seed)
    base = torch.relu(torch.randn(NB, DIM, generator=gen) + 0.3)
    gal = base.repeat(NCOPY, 1)                                    # row b + NB * j is a copy of base row b
    if eps:
        gal = torch.relu(gal + eps * torch.randn(gal.shape, generator=gen))
    mask = np.zeros((NB, NB * NCOPY), dtype=bool)
    for j in range(NCOPY):
        mask[np.arange(NB), np.arange(NB) + NB * j] = True
    return base, gal, mask, parity_terms(base, gal, "euclidean")


@pytest.fixture(scope="module")
def exact_dups():
    return scattered_copies(0.0, seed=21)


@pytest.fixture(scope="module")
def near_dups():
    return scattered_copies(NEAR_EPS, seed=22)


def dup_labels():
    """Identity b = base row b and its 32 copies; copies with j % 6 == 0 share the query's camera (junk)."""
    j = np.repeat(np.arange(NCOPY), NB)
    return (np.arange(NB, dtype=np.int64), np.tile(np.arange(NB, dtype=np.int64), NCOPY),
            np.zeros(NB, dtype=np.int64), (j % 6).astype(np.int64))


def packed_run(q, g):
    """packed_distmat on operands centred on the query mean; returns (distances, entries the contraction counted into
    its near-duplicate list)."""
    c = feature_center(q.cuda())
    qa = PackedFeatures(q.cuda(), "euclidean", False, "f16x3", c)
    gb = PackedFeatures(g.cuda(), "euclidean", False, "f16x3", c)
    out = torch.empty(q.shape[0], g.shape[0], device="cuda")
    packed_distmat(qa, gb, out)
    listed = int(engine._fixup_workspace(q.shape[0], out.device)[:8].view(torch.int64).item())
    return out.cpu().numpy(), listed


def list_capacity(Q):
    return _lib.load().ieee_distmat_fixup_bytes(Q) // 8 - 1       # (>= the entries the workspace can hold)


def test_exact_duplicates_past_fixup_capacity(cta_group, exact_dups):
    base, gal, mask, terms = exact_dups
    got, listed = packed_run(base, gal)
    assert listed == NB * NCOPY and listed > list_capacity(NB)
    bad = np.count_nonzero(got[mask] != 0.0)
    assert bad == 0, f"{bad} of {mask.sum()} duplicate distances are not 0 (max |d| {np.abs(got[mask]).max():.3g})"
    assert_distance_parity(got, base, gal, "euclidean", terms=terms)


def test_exact_duplicates_past_fixup_capacity_one_call_entry_points(exact_dups):
    base, gal, mask, terms = exact_dups
    got = compute_distance_matrix(base.cuda(), gal.cuda()).cpu().numpy()
    assert np.count_nonzero(got[mask] != 0.0) == 0
    assert_distance_parity(got, base, gal, "euclidean", terms=terms)

    qp, gp, qc, gc = dup_labels()
    ev = RetrievalEvaluator(gal.cuda(), gp, gc)
    cmc, mAP, info = ev.evaluate(base.cuda(), qp, qc, return_distmat=True, one_call=True)
    d = info["distmat"].cpu().numpy()
    assert np.count_nonzero(d[mask] != 0.0) == 0
    assert_distance_parity(d, base, gal, "euclidean", terms=terms)
    cmc_o, map_o = R.evaluate_rank(terms[0], qp, gp, qc, gc)
    assert np.array_equal(cmc, cmc_o) and abs(mAP - map_o) < 1e-9, (cmc[:3], mAP, cmc_o[:3], map_o)


def test_near_duplicates_past_fixup_capacity(cta_group, near_dups):
    base, gal, mask, terms = near_dups
    truth, _, scale, _ = terms
    got, listed = packed_run(base, gal)
    assert listed > list_capacity(NB)
    err = np.abs(got.astype(np.float64) - truth)[mask] / truth[mask]
    assert err.max() <= NEAR_BOUND, f"near-duplicate error {err.max():.3g} d (bound {NEAR_BOUND})"
    assert_distance_parity(got, base, gal, "euclidean", terms=terms)
    # the same contraction without the fix-up pass (debug bit 5): the expansion alone misses the bound
    with knob(_lib.load().ieee_set_debug_flags, 32):
        expansion, _ = packed_run(base, gal)
    err_exp = np.abs(expansion.astype(np.float64) - truth)[mask] / truth[mask]
    print(f"near duplicates: d / (|q|^2 + |g|^2) in [{(truth / scale)[mask].min():.2g}, {(truth / scale)[mask].max():.2g}]; "
          f"max error / d with fix-up {err.max():.3g}, expansion only {err_exp.max():.3g}")
    assert err_exp.max() > NEAR_BOUND


# ---------------------------------------------------------------------------------------------------------------------
# Several tiles per CTA, ragged edges, accumulation chunks, raster panels, store epilogues
# ---------------------------------------------------------------------------------------------------------------------
# (1281, 8193, 576): 363 (cta_group 1) / 198 (cta_group 2) tiles, 9 K-slices; the last pair of m tiles holds one live
# row in its first CTA and none in its peer, the last n tile one column.
RAGGED = (1281, 8193, 576)
MULTI_TILE = [(RAGGED, "euclidean"), ((1, 70001, 2304), "euclidean"),
              ((70001, 1, 64), "euclidean"),              # output pitch of 1 float: the st.global epilogue
              ((1100, 9000, 2304), "euclidean"), ((1100, 9000, 2304), "cosine")]


@pytest.fixture(scope="module")
def inputs():
    """(a, b, parity_terms) per (shape, metric, dtype), computed once for the module."""
    cache = {}

    def get(shape, metric="euclidean", dtype=torch.float32):
        key = (shape, metric, dtype)
        if key not in cache:
            a, b = features(*shape, seed=sum(shape))
            a, b = a.to(dtype), b.to(dtype)
            cache[key] = (a, b, parity_terms(a.float(), b.float(), metric))
        return cache[key]
    return get


def shape_id(s):
    return "x".join(map(str, s))


@pytest.mark.parametrize("shape,metric", MULTI_TILE, ids=[f"{shape_id(s)}-{m}" for s, m in MULTI_TILE])
def test_multi_tile_shapes(cta_group, inputs, shape, metric):
    a, b, terms = inputs(shape, metric)
    got = compute_distance_matrix(a.cuda(), b.cuda(), metric).cpu().numpy()
    assert_distance_parity(got, a, b, metric, terms=terms)


@pytest.mark.parametrize("chunk", [1, 2, 4, 5, 8, 9, 10, 0])
def test_accumulation_chunks_over_many_tiles(cta_group, inputs, chunk):
    """9 K-slices: chunk counts 9, 5 (remainder 1), 3, 2 (remainder 4), 2 (remainder 1), 1, 1; 0 = the whole-K kernel."""
    a, b, terms = inputs(RAGGED)
    with knob(_lib.load().ieee_set_accum_chunk, chunk):
        got = compute_distance_matrix(a.cuda(), b.cuda()).cpu().numpy()
        assert_distance_parity(got, a, b, "euclidean", terms=terms)     # (reads the knob: unchunked floor for 0)


@pytest.mark.parametrize("chunk", [None, 0], ids=["chunked", "whole_k"])
def test_raster_panel_does_not_change_bits(cta_group, inputs, chunk):
    """Raster order only decides which CTA computes a tile: every output's sum is the same.  At 1281 rows there are 11
    (cta_group 1) / 6 (cta_group 2) m tiles, so panels of 2 .. 5 leave a partial last panel."""
    a, b, terms = inputs(RAGGED)
    lib = _lib.load()
    outs = {}
    with accum_chunk(chunk):
        for panel in (1, 2, 3, 4, 5, 0):
            with knob(lib.ieee_set_raster_panel, panel):
                outs[panel] = compute_distance_matrix(a.cuda(), b.cuda()).cpu().numpy()
        assert_distance_parity(outs[0], a, b, "euclidean", terms=terms)
    for panel, out in outs.items():
        assert np.array_equal(out.view(np.uint32), outs[0].view(np.uint32)), f"panel {panel} differs from the default"


@pytest.mark.parametrize("chunk", [None, 0], ids=["chunked", "whole_k"])
def test_store_epilogues_give_identical_bits(cta_group, inputs, chunk):
    """G = 8193: a dense output (pitch 8193 floats) takes the st.global epilogue, a padded pitch the TMA store, and
    debug bit 2 forces st.global on the padded one.  The three compute the same fma per output."""
    a, b, terms = inputs(RAGGED)
    Q, G = a.shape[0], b.shape[0]
    lib = _lib.load()
    ac, bc = a.cuda(), b.cuda()
    with accum_chunk(chunk):
        dense = _device_distmat(ac, bc, "euclidean").cpu().numpy()
        padded = _device_distmat(ac, bc, "euclidean", out=torch.full((Q, G + 31), np.nan, device="cuda")[:, :G])
        with knob(lib.ieee_set_debug_flags, 4):
            padded_st = _device_distmat(ac, bc, "euclidean", out=torch.full((Q, G + 31), np.nan, device="cuda")[:, :G])
        padded, padded_st = (np.ascontiguousarray(t.cpu().numpy()) for t in (padded, padded_st))
        assert_distance_parity(dense, a, b, "euclidean", terms=terms)
    for name, out in (("TMA store, padded pitch", padded), ("st.global, padded pitch", padded_st)):
        assert np.array_equal(out.view(np.uint32), dense.view(np.uint32)), name


WHOLE_K_SHAPES = [RAGGED, (1100, 9000, 2304)]


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("shape", WHOLE_K_SHAPES, ids=shape_id)
def test_bf16_whole_k_over_many_tiles(cta_group, inputs, shape, metric):
    a16, b16, terms = inputs(shape, metric, torch.bfloat16)
    got = _device_distmat(a16.cuda(), b16.cuda(), metric).cpu().numpy()
    if metric == "euclidean":          # products of bf16 values are exact in fp32: the whole-K accumulator's floor
        assert_distance_parity(got, a16.float(), b16.float(), metric, floor=TC_ACCUM_FLOOR_UNCHUNKED, terms=terms)
    else:                              # normalised rows are re-rounded to bf16: bf16-level accuracy
        assert np.abs(got - terms[0]).max() < 1e-2


def assert_neg_dot_parity(got, terms, floor):
    """-(a . b) within RTOL |truth| + (reference cancellation floor + accumulator floor) (|a|^2 + |b|^2); the fp64
    truth comes from the euclidean terms of the same inputs: -(a . b) = (|a - b|^2 - |a|^2 - |b|^2) / 2."""
    dist, _, scale, _ = terms
    truth = (dist - scale) / 2
    err = np.abs(got.astype(np.float64) - truth)
    tol = RTOL * np.abs(truth) + (CANCEL_ULPS + floor) * scale
    assert (err <= tol).all(), f"max err/tol = {(err / tol).max():.3g}"


@pytest.mark.parametrize("chunk", [None, 0], ids=["chunked", "whole_k"])
@pytest.mark.parametrize("shape", WHOLE_K_SHAPES, ids=shape_id)
def test_neg_dot_over_many_tiles(cta_group, inputs, shape, chunk):
    a, b, terms = inputs(shape)
    with accum_chunk(chunk):
        got = _device_distmat(a.cuda(), b.cuda(), "neg_dot").cpu().numpy()
    assert_neg_dot_parity(got, terms, TC_ACCUM_FLOOR_UNCHUNKED if chunk == 0 else TC_ACCUM_FLOOR)
