"""ctypes binding of libieee_b200.so (include/ieee_b200.h).  No CPU fallback: a missing library or a
missing CUDA device raises, it never silently computes on the host."""
from __future__ import annotations

import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libieee_b200.so")

OK, ERR_INVALID, ERR_CUDA, ERR_WORKSPACE, ERR_NO_VALID_QUERY, ERR_SHORT_RANK_LIST, ERR_CAPACITY = range(7)
METRICS = {"euclidean": 0, "cosine": 1}
PREPARE_DEFER_JOIN, PREPARE_KEEP_CENTER = 1, 2      # flags of ieee_gallery_prepare
INTERNAL_METRICS = {"neg_dot": 2}          # -(a . b): GNN re-ranking (not a torchreid metric name)
PRECISIONS = {"f16x3": 0, "bf16": 1, "fp32_simt": 2}
DTYPES = {torch.float32: 0, torch.bfloat16: 1}

i64, i32, sz, vp, f32 = C.c_int64, C.c_int32, C.c_size_t, C.c_void_p, C.c_float


class EvalSummary(C.Structure):
    _fields_ = [("mAP", C.c_double), ("sum_ap", C.c_double), ("num_valid", i64), ("num_ties", i64),
                ("num_short", i64), ("max_rank", i32), ("status", i32), ("list_overflow", i64), ("mINP", C.c_double)]


# name -> (restype, argtypes); must list every symbol include/ieee_b200.h declares (tests/test_abi.py checks)
SIGNATURES = {
    "ieee_last_error": (C.c_char_p, []),
    "ieee_abi_version": (C.c_int, []),
    "ieee_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ieee_set_cta_group": (C.c_int, [C.c_int]),
    "ieee_launch_count": (i64, []),
    "ieee_note_launches": (i64, [i64]),
    "ieee_debug_timeline_reset": (None, []),
    "ieee_debug_timeline": (C.c_int, [C.c_char_p, sz]),
    "ieee_set_debug_flags": (C.c_int, [C.c_int]),
    "ieee_set_raster_panel": (C.c_int, [C.c_int]),
    "ieee_set_count_team": (C.c_int, [C.c_int]),
    "ieee_set_centering": (C.c_int, [C.c_int]),
    "ieee_feature_center_workspace_bytes": (sz, [i64]),
    "ieee_feature_center": (C.c_int, [vp, C.c_int, i64, i64, i64, C.c_int, i64, vp, vp, vp]),
    "ieee_set_accum_chunk": (C.c_int, [C.c_int]),
    "ieee_packed_bytes": (sz, [i64, i64, C.c_int]),
    "ieee_pack_features": (C.c_int, [vp, C.c_int, i64, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "ieee_distmat_fixup_bytes": (sz, [i64]),
    "ieee_distmat_packed": (C.c_int, [vp, i64, vp, i64, i64, C.c_int, C.c_int, vp, i64, vp, vp]),
    "ieee_distmat_workspace_bytes": (sz, [i64, i64, i64, C.c_int]),
    "ieee_distmat": (C.c_int, [vp, vp, C.c_int, i64, i64, i64, i64, i64, C.c_int, C.c_int, C.c_int, vp, i64, vp, sz, vp]),
    "ieee_gallery_group_bytes": (sz, [i64]),
    "ieee_gallery_group": (C.c_int, [vp, i64, vp, vp]),
    "ieee_rank_list_cap": (C.c_int, [vp, i64, vp, i64, vp, vp]),
    "ieee_rank_list_cap_sync": (C.c_int, [vp, i64, vp, i64, vp, C.POINTER(i32), vp]),
    "ieee_rank_gather": (C.c_int, [vp, i64, i64, i64, vp, vp, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp]),
    "ieee_rank_count_smem_bytes": (sz, [i32, i32]),
    "ieee_rank_count": (C.c_int, [vp, i64, i64, i64, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "ieee_rank_query_metrics": (C.c_int, [vp, i64, i64, i32, i32, i32, vp, vp, vp, vp, vp]),
    "ieee_rank_reduce": (C.c_int, [vp, vp, vp, i64, i32, vp, vp, vp, vp, vp]),
    "ieee_rank_finalize_workspace_bytes": (sz, [i64]),
    "ieee_rank_finalize": (C.c_int, [vp, i64, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "ieee_eval_workspace_bytes": (sz, [i64, i64, i32]),
    "ieee_eval_market1501": (C.c_int, [vp, i64, i64, i64, vp, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp]),
    "ieee_gallery_prepare_workspace_bytes": (sz, [i64]),
    "ieee_gallery_prepare": (C.c_int, [vp, i64, C.c_int, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp, i64, i64, vp, vp, vp, vp, C.c_int,
                                       vp, vp]),
    "ieee_gallery_group_join": (C.c_int, [vp]),
    "ieee_eval_market1501_f64": (C.c_int, [vp, i64, i64, i64, vp, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp]),
    "ieee_retrieve_workspace_bytes": (sz, [i64, i64, i64, C.c_int, i32]),
    "ieee_retrieve_eval": (C.c_int, [vp, i64, vp, i64, C.c_int, i64, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, i32, i32,
                                     C.POINTER(i32), vp, i64, vp, vp, vp, vp, vp, sz, vp]),
    "ieee_retrieve_prepared_workspace_bytes": (sz, [i64, i64, C.c_int, i32]),
    "ieee_retrieve_eval_prepared": (C.c_int, [vp, i64, C.c_int, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp, vp, i64, vp, vp, vp, i32, i32,
                                              C.POINTER(i32), vp, i64, vp, vp, vp, vp, vp, vp, sz, vp]),
    "ieee_topk": (C.c_int, [vp, i64, i64, i64, i64, vp, vp, vp, vp, i32, vp, vp, vp]),
    "ieee_topk_merge": (C.c_int, [vp, vp, i32, i64, i32, vp, vp, vp]),
    "ieee_gnn_rerank_workspace_bytes": (sz, [i64, i32]),
    "ieee_gnn_rerank": (C.c_int, [vp, i64, i64, i32, i32, vp, i64, vp, sz, vp]),
    "ieee_rerank_workspace_bytes": (sz, [i64, i64, i32, i32]),
    "ieee_rerank": (C.c_int, [vp, i64, vp, i64, vp, i64, i64, i64, i32, i32, C.c_double, vp, i64, vp, sz, vp]),
    "ieee_rerank_stream_workspace_bytes": (sz, [i64, i64, i32, i32]),
    "ieee_rerank_stream_scratch_bytes": (sz, [i64, i64, i32, sz]),
    "ieee_rerank_stream_prepare": (C.c_int, [vp, i64, vp, i64, i64, C.c_int, C.c_int, i32, i32, sz, vp, vp, vp, sz, vp, sz, vp]),
    "ieee_rerank_stream_block": (C.c_int, [vp, i64, i64, i32, i32, vp, i64, i64, C.c_double, vp, i64, vp, sz, vp]),
    "ieee_rerank_stream_window_workspace_bytes": (sz, [i64, i64, i32, i32, i64]),
    "ieee_rerank_stream_v_layout": (C.c_int, [i64, i64, i32, i32, C.POINTER(i64), C.POINTER(sz), C.POINTER(sz), C.POINTER(sz)]),
    "ieee_rerank_stream_pass": (C.c_int, [i32, vp, i64, vp, i64, i64, C.c_int, C.c_int, i32, i32, sz, i64, i64, i64, i64, vp, vp,
                                          vp, sz, vp, sz, vp]),
    "ieee_rerank_stream_finish": (C.c_int, [vp, sz, i64, i64, i32, i32, i64, i64, vp, vp]),
    "ieee_rerank_stream_block_window": (C.c_int, [vp, i64, i64, i32, i32, i64, vp, i64, i64, C.c_double, vp, i64, vp, sz, vp]),
    "ieee_gnn_stream_scratch_bytes": (sz, [i64, i64, i32, sz]),
    "ieee_gnn_stream_neighbours": (C.c_int, [vp, i64, vp, i64, i64, C.c_int, i32, sz, vp, vp, vp, sz, vp]),
    "ieee_gnn_stream_graph_bytes_sync": (C.c_int, [vp, i64, i64, i32, i32, vp, sz, C.POINTER(i64), vp]),
    "ieee_gnn_stream_graph": (C.c_int, [vp, vp, i64, i64, i32, i32, vp, sz, vp, sz, C.POINTER(i64), vp, vp, vp, vp, vp, vp, vp]),
    "ieee_gnn_stream_block": (C.c_int, [vp, vp, vp, vp, vp, vp, i64, i64, i64, i64, vp, i64, vp, sz, vp]),
    "ieee_gnn_stream_neighbours_rows": (C.c_int, [vp, i64, vp, i64, i64, C.c_int, i32, sz, i64, i64, i64, i64, vp, vp, vp, sz, vp]),
    "ieee_gnn_stream_layout": (C.c_int, [i64, i64, i32, i32, C.POINTER(i64), C.POINTER(sz)]),
    "ieee_gnn_stream_symbolic": (C.c_int, [vp, i64, i64, i32, i32, i64, i64, i64, i64, vp, sz, vp]),
    "ieee_gnn_stream_sizes_sync": (C.c_int, [i64, i64, i32, i32, vp, sz, C.POINTER(i64), vp]),
    "ieee_gnn_stream_numeric": (C.c_int, [i32, vp, vp, i64, i64, i32, i32, i64, i64, i64, i64, vp, sz, vp, sz, C.POINTER(i64), vp, vp,
                                          vp, vp]),
    "ieee_gnn_stream_csc": (C.c_int, [i64, i64, i32, i64, i64, i64, i64, vp, sz, vp, vp, vp, vp, vp, vp, vp]),
}

MAX_PEERS = 16


class PeerExchange(C.Structure):
    _fields_ = [("shards", i32), ("my_shard", i32), ("epoch", C.c_uint64), ("base", vp * MAX_PEERS),
                ("Qb_max", i64), ("Qb", i64), ("Qtot", i64), ("q_base", i64), ("cap", i32), ("W", i32)]


_PEER = C.POINTER(PeerExchange)
SIGNATURES.update({
    "ieee_peer_exchange_bytes": (sz, [i64, i64, i32, i32, i32]),
    "ieee_peer_alloc": (C.c_int, [sz, C.POINTER(vp), vp]),
    "ieee_peer_open": (C.c_int, [vp, C.POINTER(vp)]),
    "ieee_peer_close": (C.c_int, [vp]),
    "ieee_peer_free": (C.c_int, [vp]),
    "ieee_rank_gather_peer": (C.c_int, [vp, i64, i64, vp, vp, vp, vp, i64, vp, vp, vp, vp, _PEER, vp]),
    "ieee_rank_count_peer": (C.c_int, [vp, i64, i64, i64, vp, vp, vp, vp, _PEER, vp]),
    "ieee_rank_metrics_peer": (C.c_int, [i64, i32, vp, vp, vp, vp, _PEER, vp]),
    "ieee_peer_result_offset": (sz, [C.c_int, i64, i64, i32, i32, i32]),
    "ieee_retrieve_prepared_peer_workspace_bytes": (sz, [i64, i64, C.c_int, i32]),
    "ieee_retrieve_eval_prepared_peer": (C.c_int, [vp, i64, C.c_int, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp, vp, i64, i64, i64,
                                                   vp, vp, vp, i32, vp, i64, vp, vp, vp, vp, vp, _PEER, vp, vp, sz, vp]),
})

_lib = None


class IeeeB200Error(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"libieee_b200 error {code}: {text}")
        self.code = code
        self.text = text


def load() -> C.CDLL:
    """Load the shared library (no GPU needed just to load and inspect symbols)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m ieee_b200.build` "
                               "(nvcc, sm_100a). ieee_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(code: int) -> None:
    if code != OK:
        raise IeeeB200Error(code, load().ieee_last_error().decode())


_cuda_ok = False


def require_cuda() -> None:
    global _cuda_ok
    if _cuda_ok:
        return
    if not torch.cuda.is_available():
        raise RuntimeError("ieee_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    _cuda_ok = True


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args))
