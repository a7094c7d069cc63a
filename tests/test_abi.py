"""CPU checks of the C-ABI boundary: the library loads without a GPU and exports what the header declares."""
import ctypes
import os
import re

import pytest

from ieee_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, "include", "ieee_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ieee_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_path():
    names = header_functions()
    for required in ("ieee_distmat", "ieee_eval_market1501", "ieee_topk", "ieee_rerank", "ieee_rank_gather",
                     "ieee_rank_count", "ieee_rank_finalize", "ieee_last_error"):
        assert required in names


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    for name in header_functions():
        assert hasattr(lib, name), f"{name} declared in include/ieee_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in ieee_b200/_lib.py"
    assert sorted(_lib.SIGNATURES) == header_functions()


def test_abi_version_4_and_struct_layout():
    lib = _lib.load()
    assert lib.ieee_abi_version() == 4
    assert ctypes.sizeof(_lib.EvalSummary) == 64


def test_size_queries_need_no_gpu():
    lib = _lib.load()
    # hi + lo planes of [rows, roundup(D,64)] 16-bit plus two fp32 per row (norm, scale), 256-byte aligned sections
    assert lib.ieee_packed_bytes(128, 2304, _lib.PRECISIONS["f16x3"]) == 2 * 128 * 2304 * 2 + 1024
    assert lib.ieee_packed_bytes(128, 100, _lib.PRECISIONS["bf16"]) == 128 * 128 * 2 + 1024
    assert lib.ieee_gallery_group_bytes(15913) >= 32768 * 20 + 15913 * 8     # hash table of 2^15 slots + member lists
    assert lib.ieee_rank_finalize_workspace_bytes(1000) > 0


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="checks the no-GPU error path")
def test_no_cpu_fallback():
    import torch
    from ieee_b200.metrics import compute_distance_matrix, evaluate_rank
    lib = _lib.load()
    sm, cc = ctypes.c_int(), ctypes.c_int()
    assert lib.ieee_device_info(ctypes.byref(sm), ctypes.byref(cc)) == _lib.ERR_CUDA
    assert b"no CPU fallback" in lib.ieee_last_error()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        compute_distance_matrix(torch.rand(4, 8), torch.rand(5, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        evaluate_rank(torch.rand(4, 5).numpy(), [1] * 4, [1] * 5, [0] * 4, [1] * 5)
    # argument errors keep the reference's exception types even without a GPU (distance.py:26-44)
    with pytest.raises(ValueError):
        compute_distance_matrix(torch.rand(4, 8), torch.rand(5, 8), "manhattan")
    with pytest.raises(AssertionError):
        compute_distance_matrix(torch.rand(4, 8), torch.rand(5, 9))


def test_patch_torchreid_rebinds_the_three_call_sites(monkeypatch):
    """ieee_b200.patch_torchreid(): the names the fork's engine imported (engine.py:18-19, utils/__init__.py:4)."""
    import sys
    import types

    import ieee_b200
    from ieee_b200.metrics import distance, rank
    from ieee_b200.utils import rerank

    fake_engine = types.ModuleType("torchreid.engine.engine")
    fake_engine.compute_distance_matrix = fake_engine.evaluate_rank = fake_engine.re_ranking = object()
    fake_utils = types.ModuleType("torchreid.utils")
    fake_utils.re_ranking = object()
    monkeypatch.setitem(sys.modules, "torchreid", types.ModuleType("torchreid"))
    monkeypatch.setitem(sys.modules, "torchreid.engine.engine", fake_engine)
    monkeypatch.setitem(sys.modules, "torchreid.utils", fake_utils)
    for name in ("torchreid.metrics.distance", "torchreid.metrics.rank", "torchreid.utils.rerank"):
        monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
    ieee_b200.patch_torchreid()
    assert fake_engine.compute_distance_matrix is distance.compute_distance_matrix
    assert fake_engine.evaluate_rank is rank.evaluate_rank
    assert fake_engine.re_ranking is rerank.re_ranking and fake_utils.re_ranking is rerank.re_ranking
    assert sys.modules["torchreid.metrics.rank"] is rank and sys.modules["torchreid.metrics.distance"] is distance


def test_signatures_match_the_reference():
    """Same parameter names and defaults as distance.py:6, rank.py:246-255 and rerank.py:31."""
    import inspect

    from ieee_b200.metrics import compute_distance_matrix, evaluate_rank
    from ieee_b200.utils import re_ranking

    p = inspect.signature(compute_distance_matrix).parameters
    assert list(p)[:3] == ["input1", "input2", "metric"] and p["metric"].default == "euclidean"
    p = inspect.signature(evaluate_rank).parameters
    assert list(p) == ["distmat", "q_pids", "g_pids", "q_camids", "g_camids", "max_rank", "use_metric_cuhk03", "use_cython"]
    assert (p["max_rank"].default, p["use_metric_cuhk03"].default, p["use_cython"].default) == (20, False, True)
    p = inspect.signature(re_ranking).parameters
    assert list(p) == ["q_g_dist", "q_q_dist", "g_g_dist", "k1", "k2", "lambda_value"]
    assert (p["k1"].default, p["k2"].default, p["lambda_value"].default) == (20, 6, 0.3)


def test_shipped_library_is_tcgen05_tma_code_for_sm100a_only():
    """The contraction kernels of the built .so are tcgen05 / TMEM / TMA code (UTCHMMA, LDTM, UTMALDG, UTMASTG in SASS),
    there is no legacy mma.sync (HMMA / IMMA) anywhere, and sm_100a is the only architecture in the file."""
    import re
    import shutil
    import subprocess
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    _lib.load()
    txt = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert set(re.findall(r"arch = (sm_\w+)", txt)) == {"sm_100a"}
    ops_by_fn = {}
    for m in re.finditer(r"Function : (\S+)\n(.*?)(?=\n\s*Function : |\Z)", txt, re.S):
        ops_by_fn[m.group(1)] = set(re.findall(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)", m.group(2), re.M))
    gemm = {k: v for k, v in ops_by_fn.items() if "distmat_umma" in k}
    assert len(gemm) >= 4
    for name, ops in gemm.items():
        assert {"UTCHMMA", "LDTM", "UTMALDG", "UTCBAR"} <= ops, (name, sorted(ops))
    assert any("UTMASTG" in ops for ops in gemm.values())
    legacy = {k for k, ops in ops_by_fn.items() if ops & {"HMMA", "IMMA", "DMMA"}}
    assert not legacy, legacy
