"""Device-resident evaluation: the reference's ``Engine._evaluate`` tail (torchreid/engine/engine.py:391-425)
without its host round trips.

The reference concatenates features on the CPU (engine.py:368-373), normalises (:391-394), builds the whole
Q x G matrix with torch CPU (:399-400), optionally re-ranks (:402-406) and calls ``evaluate_rank`` (:410-417).
Here features stay in HBM, the gallery is packed and grouped once, queries are processed in blocks whose
distance block lives only in HBM scratch, and -- when the process group has more than one rank -- every rank
owns a contiguous slice of the gallery: relevant-pair distances are all-gathered, integer rank counts are
all-reduced, and every rank ends with the same (cmc, mAP) the single-GPU path produces.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from .metrics.rank import GalleryLabels, RankStages, _as_device, copy_stream, raise_for_status
from .peer import PeerLink, link_for
from .utils.rerank import re_ranking_device

DEFAULT_BLOCK_BYTES = 4 << 30   # HBM scratch for one distance block


class Trace:
    """CUDA-event timeline of one evaluation (IEEE_B200_TRACE=1): mark() records an event on the current stream,
    report() -- after a synchronize -- lists the GPU time of every mark relative to the first and the host time at
    which it was enqueued.  The reference only has wall-clock AverageMeters (engine.py:365-367)."""

    def __init__(self):
        import os
        self.enabled = os.environ.get("IEEE_B200_TRACE", "0") == "1"
        self.marks = []

    def mark(self, name: str):
        if self.enabled:
            import time
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.marks.append((name, ev, time.perf_counter()))

    def report(self):
        if not self.enabled or not self.marks:
            return
        torch.cuda.synchronize()
        _, e0, t0 = self.marks[0]
        for name, ev, t in self.marks:
            print("[trace] %-28s gpu %8.3f ms   enqueued at %8.3f ms" % (name, e0.elapsed_time(ev), (t - t0) * 1e3))
        self.marks = []


TRACE = Trace()

# List-capacity memo.  The per-query list capacity (largest identity group among the queried ids) sizes buffers and
# shared memory, and finding it costs a host round trip (plus, with several ranks, a collective that has to line the
# ranks up in the middle of a step).  It only depends on the label tensors, so it is remembered per
# (gallery ids, query ids) tensor identity AND version counter: handing in the same, unmodified tensors again skips the
# query.  It is a hint, not a trusted value: the gather kernel flags any list that does not fit, and evaluate()
# then recomputes the capacity and runs again.
_CAP_MEMO = {}
# The key is built from tensor identities (address, size, version counter), so every entry also KEEPS its key
# tensors alive: a freed label tensor whose address is reused by another tensor of the same size could otherwise
# produce a false hit -- harmless on one GPU (the overflow flag catches it), but with several ranks a hit on one
# rank and a miss on another would make them issue different collectives.
_CAP_MEMO_REFS = {}


def _memo_put(key, value, refs):
    if len(_CAP_MEMO) > 64:
        _CAP_MEMO.clear()
        _CAP_MEMO_REFS.clear()
    _CAP_MEMO[key] = value
    _CAP_MEMO_REFS[key] = refs


def _memo_drop(key):
    _CAP_MEMO.pop(key, None)
    _CAP_MEMO_REFS.pop(key, None)


_STAGE_POOL = {}


def _stages_for(Qb, cap, world, device, width=0):
    """Stage buffers are reused across evaluations of the same shape (all work on them is ordered by the compute
    stream); creating the dozen small tensors costs more host time than the kernels take to launch."""
    key = (Qb, cap, world, str(device), width)
    st = _STAGE_POOL.get(key)
    if st is None:
        if len(_STAGE_POOL) > 8:
            _STAGE_POOL.clear()
        st = _STAGE_POOL[key] = RankStages(Qb, cap, world, device, width)
    return st


_ONE_CALL_POOL = {}
_RESULT_HOST = {}


def _one_call_buffers(key, ws_bytes, res_bytes, device):
    """Workspace and result block of a one-call evaluation, reused per key (stream-ordered like the stage pool).  The
    result block is zeroed once, here: the one-GPU entry point never writes its stats words."""
    buf = _ONE_CALL_POOL.get(key)
    if buf is None:
        if len(_ONE_CALL_POOL) > 8:
            _ONE_CALL_POOL.clear()
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=device)
        buf = _ONE_CALL_POOL[key] = (ws, torch.zeros(res_bytes, dtype=torch.uint8, device=device))
    return buf


def _read_result(res: torch.Tensor):
    """One device->host copy of a result block [stats int64[4] | summary (64 B) | cmc float32[K']] into a pooled pinned
    buffer, then a stream synchronise.  stats = [gather overflow = needed capacity (0: all lists fitted), tie pairs,
    longest merged list, pad].  Returns ((overflow, longest), summary, cmc); the overflow is also taken from the
    summary, where the one-GPU one-call entry point reports it."""
    key = (str(res.device), res.numel())
    host = _RESULT_HOST.get(key)
    if host is None:
        host = _RESULT_HOST[key] = torch.empty(res.numel(), dtype=torch.uint8, pin_memory=True)
    host.copy_(res, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return _parse_result(host.numpy())


def _parse_result(out: np.ndarray):
    """((overflow, longest), summary, cmc) from the host copy of a result block (see _read_result); cmc is a copy."""
    overflow, _, longest = (int(v) for v in out[:32].view(np.int64)[:3])
    summary = _lib.EvalSummary.from_buffer_copy(out[32:96].tobytes())
    return (overflow or summary.list_overflow, longest), summary, out[96:].view(np.float32).copy()


def _features_key(t: torch.Tensor):
    return (t.data_ptr(), t._version, tuple(t.shape), t.stride(0), t.dtype)


def _tensor_key(t):
    return (t.data_ptr(), t.numel(), t._version, str(t.device)) if isinstance(t, torch.Tensor) else None


def shard_bounds(num_rows: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous gallery slice of ``rank``: [start, stop).  Global index = local index + start, so the
    (distance, index) tie order is the same as on one GPU."""
    base, rem = divmod(num_rows, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def rerank_owned(Q: int, G: int, world: int, rank: int) -> tuple[int, int, int, int]:
    """Samples whose strips ``rank`` computes when ``world`` ranks prepare k-reciprocal re-ranking together: queries
    [q0, q1) and gallery rows [g0, g1).  Each segment is cut into 256-sample strips, dealt out as shard_bounds deals
    rows: every range starts at a multiple of 256 of its segment, and ranks differ by at most one strip per segment."""
    def split(n):
        a, b = shard_bounds((n + 255) // 256, world, rank)
        return min(n, 256 * a), min(n, 256 * b)
    return split(Q) + split(G)


def rerank_ranges(offsets: list[int], G: int) -> list[tuple[int, int]]:
    """Gallery rows [a, b) whose columns each rank computes in the strips when ranks holding slices that start at
    ``offsets`` (rank order, tiling [0, G)) prepare k-reciprocal re-ranking together: a is the rank's slice start rounded
    up to a multiple of 256 (0 for the first rank), b the next rank's a (G for the last).  The ranges tile [0, G) in rank
    order and start at multiples of 256, where the contraction puts a column as it does for the whole gallery; a range
    is empty when its slice holds no such start, and reaches up to 255 rows into the slices after its own."""
    a = [0] + [min(G, (o + 255) // 256 * 256) for o in offsets[1:]]
    return [(a[r], a[r + 1] if r + 1 < len(a) else G) for r in range(len(a))]


def centering_applies(metric: str, precision: str) -> bool:
    """Euclidean operands are packed relative to a common centre (ieee_pack_features); cosine is not translation
    invariant and the 1-pass bf16 mode multiplies bf16 inputs exactly as they are."""
    return metric == "euclidean" and precision != "bf16" and _lib.load().ieee_set_centering(-1) != 0


def feature_center(feats: torch.Tensor, normalize: bool = False, max_rows: int = 0) -> torch.Tensor:
    """Column mean over a strided sample of the rows (unit length when the rows will be normalised): float32 [D] on
    the device, deterministic (ieee_feature_center)."""
    assert feats.is_cuda and feats.dim() == 2 and feats.dtype in _lib.DTYPES and feats.shape[0] > 0
    if feats.stride(1) != 1:
        feats = feats.contiguous()
    rows, D = feats.shape
    lib = _lib.load()
    center = torch.empty(D, dtype=torch.float32, device=feats.device)
    ws = torch.empty(lib.ieee_feature_center_workspace_bytes(D), dtype=torch.uint8, device=feats.device)
    with torch.cuda.device(feats.device):
        _lib.call("ieee_feature_center", feats.data_ptr(), _lib.DTYPES[feats.dtype], feats.stride(0), rows, D, int(normalize),
                  max_rows, center.data_ptr(), ws.data_ptr(), _lib.stream())
    return center


class PackedFeatures:
    """Feature rows in the operand layout of the tensor-core kernel (ieee_pack_features)."""

    def __init__(self, feats: torch.Tensor, metric: str, normalize: bool, precision: str, center: torch.Tensor | None = None):
        if not (feats.is_cuda and feats.dim() == 2):
            raise TypeError("PackedFeatures: expected a 2-D CUDA tensor")
        if feats.dtype not in _lib.DTYPES:
            raise TypeError("PackedFeatures: features must be float32 or bfloat16, got {}".format(feats.dtype))
        if feats.stride(1) != 1:
            feats = feats.contiguous()
        self._allocate(*feats.shape, metric, precision, center, feats.device)
        if self.rows:
            _lib.call("ieee_pack_features", feats.data_ptr(), _lib.DTYPES[feats.dtype], feats.stride(0), self.rows, self.D,
                      self.metric, int(normalize), self.precision, _lib.ptr(center), self.buf.data_ptr(), _lib.stream())

    @classmethod
    def _empty(cls, rows: int, D: int, metric: str, precision: str, center: torch.Tensor | None, device):
        """The buffer of `rows` packed rows, left for the caller to fill (ieee_gallery_prepare)."""
        pk = cls.__new__(cls)
        pk._allocate(rows, D, metric, precision, center, device)
        return pk

    def _allocate(self, rows, D, metric, precision, center, device):
        self.rows, self.D = rows, D
        self.metric = _lib.METRICS[metric] if metric in _lib.METRICS else _lib.INTERNAL_METRICS[metric]
        self.precision = _lib.PRECISIONS[precision]
        self.center = center
        self.buf = torch.empty(max(_lib.load().ieee_packed_bytes(rows, D, self.precision), 256), dtype=torch.uint8,
                               device=device)


def packed_distmat(q: PackedFeatures, g: PackedFeatures, out: torch.Tensor) -> torch.Tensor:
    assert q.D == g.D and q.metric == g.metric and q.precision == g.precision
    assert _lib.ptr(q.center) == _lib.ptr(g.center), "both operands must be packed with the same centre"
    _lib.call("ieee_distmat_packed", q.buf.data_ptr(), q.rows, g.buf.data_ptr(), g.rows, q.D, q.metric, q.precision,
              out.data_ptr(), out.stride(0), _fixup_workspace(q.rows, out.device).data_ptr(), _lib.stream())
    return out


_FIXUP_WS = {}


def _fixup_workspace(rows: int, device) -> torch.Tensor:
    """Near-duplicate list of the contraction (ieee_distmat_fixup_bytes): one per device and stream, grown on demand;
    contractions on one stream run one after the other, so they can share it."""
    key = (str(device), torch.cuda.current_stream(device).cuda_stream)
    need = _lib.load().ieee_distmat_fixup_bytes(rows)
    ws = _FIXUP_WS.get(key)
    if ws is None or ws.numel() < need:
        ws = _FIXUP_WS[key] = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=device)
    return ws


def _as_features(t: torch.Tensor) -> torch.Tensor:
    """float32 / bfloat16 features pass through; float16 (AMP extraction) and float64 are computed in float32, as
    compute_distance_matrix does -- there is no float64 contraction and no gradient on this path."""
    if not isinstance(t, torch.Tensor) or t.dim() != 2:
        raise TypeError("features must be a 2-D torch.Tensor")
    if t.dtype in _lib.DTYPES:
        return t.detach()
    if t.dtype in (torch.float16, torch.float64):
        return t.detach().float()
    raise TypeError("features must be a floating point tensor, got {}".format(t.dtype))


class RetrievalEvaluator:
    """distmat -> rank -> CMC/mAP over a (possibly sharded) gallery.

    ``gf, g_pids, g_camids`` are THIS rank's gallery slice (the whole gallery when ``group`` is None);
    ``g_offset`` its first global row and ``g_total`` the gallery size over all ranks.

    ``rerank=True`` ranks k-reciprocal re-ranked distances (rerank.py:31-113 with ``k1``, ``k2``, ``lambda_value``;
    k1, k2 default to 20, 6) instead of the plain ones, with the same bits as ``re_ranking`` on the three distance
    matrices, but without any N x N matrix (N = queries + gallery): the re-ranking state is prepared from the features
    in column strips (ieee_rerank_stream_prepare, strips sized by ``block_bytes``) and each query block's distances are
    re-ranked before they are ranked.  The gallery must be in HBM (not ``from_host``).

    With ``group`` (a torch.distributed process group; NCCL for device tensors) and ``rerank=True`` the re-ranking is
    over the whole sharded gallery, with the bits of one GPU holding it all: every rank returns what a one-GPU
    ``rerank=True`` evaluator returns (ieee_rerank_stream_pass / _finish / _block_window).  The slices must tile
    [0, g_total) in rank order (checked once, collectively; ValueError on every rank otherwise).  No rank holds the
    whole gallery: the ranks compute every strip of the prepare call together, each the columns of its share of the
    queries (rerank_owned) and of its gallery range (rerank_ranges: its slice, 256-aligned, so up to 255 rows of the
    next slices are sent to it once).  A gallery strip's rows are exchanged for that strip alone, and the strips' small
    results (column maxima, neighbour lists, the k-reciprocal weights' inputs) are reduced across the ranks; the ranks
    share one strip width, the narrowest their ``block_bytes`` allow.  What stays is sized by this rank's slice of Gs rows:
    about 8 (k1+1)(round(k1/2)+2) bytes per sample of the whole set plus k2 times that per query and per slice row
    (2 KB * N + 24 KB * (Q + Gs) at k1 = 20, k2 = 6), plus ``block_bytes``.  The plain sharded path's condition for
    the bits of one GPU applies to the query blocks' own distances (this rank's contraction against its slice).

    ``rerank="gnn"`` ranks the GNN re-ranked similarity (gnn_reranking.py:27-59; k1, k2 default to 26, 7, the reference
    driver's values), negated so that it ranks as a distance: what ``gnn_reranking_distmat`` computes on the
    evaluator's features.  The score is X X^T of the features after ``normalize_feature``, packed with the negative dot
    product and no centre; ``dist_metric`` and ``lambda_value`` are not used.  The adjacency is held sparse
    (ieee_gnn_stream_*: neighbours from row strips sized by ``block_bytes``, then A as CSR rows and an inverted index of
    its gallery rows), and a query block's distances come from it instead of a contraction.  Same limits on the
    gallery as ``rerank=True``, and no ``group``; 1 <= k2 <= k1 <= min(N, 1024).

    With ``query_group`` (a torch.distributed process group, NCCL) and ``rerank="gnn"``, the ranks of the group share
    the GNN re-ranking: every rank holds the whole gallery (``gf``, ``g_pids``, ``g_camids``) and is handed the whole
    query set, and every rank returns what an evaluator without ``query_group`` returns, bit for bit (cmc, mAP, ap,
    first, mINP and ``ranked_lists`` of all queries).  Each rank owns the queries and gallery rows rerank_owned(Q, G,
    world, rank) gives: it computes those rows of every stage whose work grows as N^2 (neighbour lists, the symbolic
    counts, the rows of the adjacency's structures, the sort of the same columns of the CSC) and evaluates its own
    queries; the stages linear in the adjacency's entries run on every rank (ieee_gnn_stream_neighbours_rows /
    _symbolic / _sizes_sync / _numeric / _csc).  The per-query results are all-gathered and reduced on every rank.
    ``return_distmat=True`` returns this rank's own query rows only: rows [q0, q1) of the queries, (q0, q1) =
    rerank_owned(Q, G, world, rank)[:2] (possibly none).  This buys time, not memory: while the state is built every rank
    holds B1, A1, B2 and the CSC whole, as one GPU does.  The ranks must agree on G, D, dtype, precision,
    normalize_feature, k1 and k2 (checked once at construction) and on the number of queries (checked by every
    evaluate); ValueError on every rank otherwise.  ``query_group`` cannot be combined with ``group``, and plain and
    k-reciprocal evaluation take ``group`` instead.
    """

    def __init__(self, gf: torch.Tensor, g_pids, g_camids, dist_metric: str = "euclidean", normalize_feature: bool = False,
                 precision: str | None = None, max_rank: int = 20, group=None, g_offset: int = 0, g_total: int | None = None,
                 block_bytes: int = DEFAULT_BLOCK_BYTES, center: torch.Tensor | None = None, exchange: str | None = None,
                 rerank: bool | str = False, k1: int | None = None, k2: int | None = None, lambda_value: float = 0.3,
                 query_group=None):
        _lib.require_cuda()
        if dist_metric not in _lib.METRICS:
            raise ValueError('Unknown distance metric: {}. Please choose either "euclidean" or "cosine"'.format(dist_metric))
        if isinstance(rerank, str) and rerank != "gnn":
            raise ValueError('rerank must be False, True or "gnn", got {!r}'.format(rerank))
        self.device = gf.device if gf is not None else torch.device("cuda", torch.cuda.current_device())
        self.gnn = rerank == "gnn"
        # GNN re-ranking scores with the negative dot product whatever the distance metric (gnn_reranking.py:31)
        self.metric, self.normalize = ("neg_dot" if self.gnn else dist_metric), normalize_feature
        self.precision = precision or ("bf16" if gf is not None and gf.dtype == torch.bfloat16 else "f16x3")
        self.rerank = bool(rerank)
        if query_group is not None:
            self._check_query_group(query_group, group)
        if k1 is None:
            k1 = 26 if self.gnn else 20
        if k2 is None:
            k2 = 7 if self.gnn else 6
        if self.rerank:
            self._check_rerank(gf, group, k1, k2, g_total)
        self.k1, self.k2, self.lambda_value = k1, k2, float(lambda_value)
        self._rr = None          # re-ranking state of the last query set (_rerank_prepare)
        self._rr_scratch = None  # the blend's accumulators, one block
        self.max_rank = max_rank
        self.group = group
        self.world = 1 if group is None else torch.distributed.get_world_size(group)
        self.g_offset = g_offset
        self.block_bytes = block_bytes
        # how the ranks of a sharded gallery exchange lists and counts: "peer" = stores into NVLink peer memory from
        # inside the rank kernels (NCCL process groups), "nccl" = all-gather + all-reduce launches (any backend)
        self.exchange = exchange or os.environ.get("IEEE_B200_EXCHANGE") or (
            "peer" if self.world > 1 and torch.distributed.get_backend(group) == "nccl" else "nccl")
        if gf is not None:
            gf = _as_features(gf)
        # Euclidean operands are packed relative to a common centre (PackedFeatures).  It is taken from the QUERY set:
        # queries are replicated on every rank of a sharded gallery, so all shards -- and a single-GPU evaluation of
        # the same queries -- derive the same vector without exchanging anything.  The gallery is therefore packed
        # on the first evaluate(), or here when the caller hands a centre in.
        self._use_center = not self.gnn and centering_applies(dist_metric, self.precision)
        self.center = center
        self._gallery_dev = gf
        # the gallery as packed row chunks [(first row, PackedFeatures)]: one chunk when the features are already
        # in HBM, several when they are streamed from the host (from_host) so that the contraction of chunk i
        # overlaps the PCIe copy of chunk i + 1
        self.chunks = []
        with torch.cuda.device(self.device):
            # a device-resident gallery is prepared by ONE foreign call (grouping on a side stream beside centre + pack):
            # here when no centre is needed or one was handed in, else in the first evaluate()
            self.labels = GalleryLabels(g_pids, g_camids, self.device, build=gf is None)
            if gf is not None and (not self._use_center or center is not None):
                self._prepare_gallery(None)
        self.G = self.labels.G
        self.g_total = self.G if g_total is None else g_total
        self._block = None
        self._early_q = None
        self._copy = None
        self._host_gallery = None
        self._label_keys = (_tensor_key(g_pids), _tensor_key(g_camids))
        self._label_refs = (g_pids, g_camids)
        self._slices = self._gallery_slices() if self.rerank and group is not None else None
        self.query_group = query_group
        if query_group is not None:
            self._q_world = torch.distributed.get_world_size(query_group)
            self._q_rank = torch.distributed.get_rank(query_group)
            self._check_ranks_agree(gf)

    def _check_query_group(self, query_group, group):
        if not (torch.distributed.is_available() and isinstance(query_group, torch.distributed.ProcessGroup)):
            raise ValueError("query_group must be a torch.distributed process group, got {!r}".format(type(query_group).__name__))
        if group is not None:
            raise ValueError("query_group (every rank holds the whole gallery) cannot be combined with group (a sharded "
                             "gallery)")
        if not self.gnn:
            raise ValueError('query_group shares GNN re-ranking (rerank="gnn") only: plain and k-reciprocal evaluation run '
                             "on several GPUs over a sharded gallery with group=")

    def _check_ranks_agree(self, gf):
        """One all-gather at construction: every rank of query_group must hold the same gallery shape and settings (not
        block_bytes: the bits depend on neither strip width nor block size).  ValueError on every rank otherwise."""
        import torch.distributed as dist_
        mine = [self.G, gf.shape[1], _lib.DTYPES[gf.dtype], _lib.PRECISIONS[self.precision], int(self.normalize), self.k1, self.k2]
        with torch.cuda.device(self.device):
            every = torch.empty((self._q_world, len(mine)), dtype=torch.int64, device=self.device)
            dist_.all_gather_into_tensor(every, torch.tensor(mine, dtype=torch.int64, device=self.device), group=self.query_group)
            every = every.cpu().tolist()
        if any(e != every[0] for e in every):
            raise ValueError("query_group: the ranks disagree on (G, D, dtype, precision, normalize_feature, k1, k2): "
                             "{}".format([tuple(e) for e in every]))

    def _agree_on_queries(self, qf: torch.Tensor):
        """One all-gather per evaluation of a query_group: the ranks must hold the same number of queries (ValueError on
        every rank otherwise), and when any rank has no GNN state for these queries, every rank prepares it anew, so that
        all of them take part in the same exchanges."""
        import torch.distributed as dist_
        key = (_features_key(qf), self.k1, self.k2)
        fresh = int(self._rr is None or self._rr["key"] != key)
        every = torch.empty((self._q_world, 2), dtype=torch.int64, device=self.device)
        dist_.all_gather_into_tensor(every, torch.tensor([qf.shape[0], fresh], dtype=torch.int64, device=self.device),
                                     group=self.query_group)
        every = every.cpu().tolist()
        if any(q != every[0][0] for q, _ in every):
            raise ValueError("query_group: the ranks hold different numbers of queries: {}".format([q for q, _ in every]))
        if any(f for _, f in every):
            self._rr = None

    def _query_range(self, Q: int) -> tuple[int, int]:
        """Queries [q0, q1) this rank evaluates: its own (rerank_owned) with a query_group, else all of them."""
        return rerank_owned(Q, self.G, self._q_world, self._q_rank)[:2] if self.query_group is not None else (0, Q)

    def _gallery_slices(self):
        """[(g_offset, rows, block_bytes)] of every rank, all-gathered once.  Every rank gets the same list and so reaches
        the same verdict: slices that do not tile [0, g_total) in rank order raise ValueError on every rank.  From the
        block_bytes of all ranks every rank derives the same strip width."""
        import torch.distributed as dist_
        with torch.cuda.device(self.device):
            mine = torch.tensor([self.g_offset, self.G, self.g_total, self.block_bytes], dtype=torch.int64, device=self.device)
            every = torch.empty((self.world, 4), dtype=torch.int64, device=self.device)
            dist_.all_gather_into_tensor(every.view(-1), mine, group=self.group)
            every = every.cpu().tolist()
        total = every[0][2]
        starts = [sum(e[1] for e in every[:r]) for r in range(self.world)]
        if any(e[0] != s or e[2] != total for e, s in zip(every, starts)) or starts[-1] + every[-1][1] != total:
            raise ValueError("rerank=True over a sharded gallery: the slices (g_offset, rows, g_total) of the ranks {} do "
                             "not tile [0, g_total) in rank order".format([tuple(e[:3]) for e in every]))
        return [(off, rows, bb) for off, rows, _, bb in every]

    def _check_rerank(self, gf, group, k1, k2, g_total):
        mode = 'rerank="gnn"' if self.gnn else "rerank=True"
        if group is not None and self.gnn:
            raise ValueError("{} needs the whole gallery on one GPU: re-ranking over a sharded gallery (group) "
                             "is not supported".format(mode))
        if group is not None and not (torch.distributed.is_available() and isinstance(group, torch.distributed.ProcessGroup)):
            raise ValueError("rerank=True over a sharded gallery needs a torch.distributed process group as group, "
                             "got {!r}".format(type(group).__name__))
        if gf is None:
            raise ValueError("{} needs the gallery features on the device: from_host streams them from the host".format(mode))
        if self.precision not in ("f16x3", "bf16"):
            raise ValueError("{} computes with the tensor-core precisions f16x3 and bf16, not {}".format(mode, self.precision))
        if not all(isinstance(k, (int, np.integer)) and not isinstance(k, bool) for k in (k1, k2)):
            raise ValueError("{}: k1 and k2 must be integers, got k1={!r} k2={!r}".format(mode, k1, k2))
        if self.gnn:
            if not 1 <= k2 <= k1 <= 1024:
                raise ValueError('rerank="gnn" needs 1 <= k2 <= k1 <= min(N, 1024), got k1={} k2={}'.format(k1, k2))
            # the library's size query states the other limits (N <= 2^20), here for the fewest queries that give k1
            # samples; the first evaluate() checks k1 <= N with the real query count
            G = max(gf.shape[0], 1)
            if _lib.load().ieee_gnn_stream_scratch_bytes(max(1, k1 - G), G, k1, 0) == 0:
                raise ValueError('rerank="gnn": ' + _lib.load().ieee_last_error().decode())
            return
        # the library's size query states its limits (k1 + 1 <= 512, k2 <= k1 + 1, the expansion's sort, N < 2^24), here
        # for the fewest queries that give k1 + 1 samples; evaluate() checks k1 + 1 <= N with the real query count
        G = max(gf.shape[0] if g_total is None else g_total, 1)
        if _lib.load().ieee_rerank_stream_workspace_bytes(max(1, k1 + 1 - G), G, k1, k2) == 0:
            raise ValueError("rerank=True: " + _lib.load().ieee_last_error().decode())

    def _rerank_prepare(self, qf: torch.Tensor):
        """Re-ranking state of this query set (ieee_rerank_stream_prepare, or the ieee_gnn_stream_* calls): kept while
        the same, unmodified query tensor is evaluated again with the same k1 and k2."""
        k1, k2 = self.k1, self.k2
        key = (_features_key(qf), k1, k2)
        if self._rr is not None and self._rr["key"] == key:
            return self._rr
        # the previous state, the distance block and the blend's accumulators are free while the strips are computed:
        # the block budget (block_bytes) then covers the strips, and later the block and its accumulators
        self._rr = self._block = self._rr_scratch = None
        if self.gnn:
            self._rr = self._gnn_prepare(qf, key)
            return self._rr
        Q, D = qf.shape
        G = self.g_total
        if k1 + 1 > Q + G:
            raise ValueError("rerank=True: k1 + 1 = {} exceeds the {} query and gallery samples".format(k1 + 1, Q + G))
        lib = _lib.load()
        ws_bytes = lib.ieee_rerank_stream_window_workspace_bytes(Q, G, k1, k2, self.G)
        # (a sharded prepare sizes its own scratch for its part of the strips)
        sc_bytes = lib.ieee_rerank_stream_scratch_bytes(Q, G, k1, self.block_bytes) if self.group is None else 1
        if ws_bytes == 0 or sc_bytes == 0:
            raise ValueError("rerank=True: " + lib.ieee_last_error().decode())
        qpk = self._take_early_q(qf)
        if qpk is None:
            qpk = PackedFeatures(qf, self.metric, self.normalize, self.precision, self.center)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        if self.group is None:
            strips = torch.empty(sc_bytes, dtype=torch.uint8, device=self.device)    # released (stream-ordered) on return
        colmax = torch.empty(Q + G, dtype=torch.float32, device=self.device)
        rank = torch.empty((Q + G, k1 + 1), dtype=torch.int32, device=self.device)
        if self.group is None:
            _lib.call("ieee_rerank_stream_prepare", qpk.buf.data_ptr(), Q, self.chunks[0][1].buf.data_ptr(), G, D, qpk.metric,
                      qpk.precision, k1, k2, self.block_bytes, colmax.data_ptr(), rank.data_ptr(), ws.data_ptr(), ws_bytes,
                      strips.data_ptr(), sc_bytes, _lib.stream())
        else:
            self._rerank_prepare_sharded(qpk, colmax, rank, ws)
        TRACE.mark("re-ranking state prepared")
        # qf is kept so that its address cannot be reused by another tensor while the key refers to it; k1 and k2
        # fix the workspace's layout, so the block calls take them from here
        self._rr = {"key": key, "qf": qf, "Q": Q, "k1": k1, "k2": k2, "packed": qpk, "ws": ws, "colmax": colmax,
                    "rank": rank}
        return self._rr

    def _rerank_prepare_sharded(self, qpk: PackedFeatures, colmax, rank, ws):
        """The prepare call's passes with every strip computed by all ranks together, each the part of every strip row in
        its columns: its share of the queries (rerank_owned) and its gallery range (rerank_ranges), packed once.  Per strip
        of pass 0 the part's column maxima are all-reduced (MAX), and the part's two top-(k1+1) lists all-gathered and
        merged into `rank`; pass 1 writes V's membership of all rows from `rank`, then per strip the members' values in the
        part, summed across the ranks (int32: one non-zero contributor each) and weighed.  A gallery strip's rows are
        summed from the slices that hold them (zeros elsewhere) and packed by every rank.  The finish covers this rank's
        slice."""
        import torch.distributed as dist_
        Q, G, k1, k2, D = qpk.rows, self.g_total, self.k1, self.k2, qpk.D
        lib, dev, stream, k1p = _lib.load(), self.device, _lib.stream(), k1 + 1
        me, world = dist_.get_rank(self.group), self.world
        ranges = rerank_ranges([off for off, _, _ in self._slices], G)
        parts = [rerank_owned(Q, G, world, r)[:2] + ranges[r] for r in range(world)]
        W = min(lib.ieee_rerank_stream_part_width(Q, G, k1, *part, bb) for part, (_, _, bb) in zip(parts, self._slices))
        part = parts[me]
        sc_bytes = lib.ieee_rerank_stream_part_scratch_bytes(Q, G, k1, *part, W) if W else 0
        if sc_bytes == 0:
            raise ValueError("rerank=True: " + lib.ieee_last_error().decode())
        scratch = torch.empty(sc_bytes, dtype=torch.uint8, device=dev)         # released (stream-ordered) on return
        gpart = self._gallery_range(ranges)
        TRACE.mark("re-ranking: gallery range packed")
        cap, off_col, off_val, off_cnt = C.c_int64(), C.c_size_t(), C.c_size_t(), C.c_size_t()
        _lib.call("ieee_rerank_stream_v_layout", Q, G, k1, k2, C.byref(cap), C.byref(off_col), C.byref(off_val), C.byref(off_cnt))
        v_val = ws[off_val.value: off_val.value + 4 * (Q + G) * cap.value].view(torch.int32).view(Q + G, cap.value)
        gf, off = self._gallery_dev, self.g_offset
        raw = torch.empty((W, D), dtype=gf.dtype, device=dev)                   # a gallery strip's rows
        lists = torch.empty((2, 2 * W * k1p), dtype=torch.int32, device=dev)    # this rank's lists: indices, value bits
        every = torch.empty((2, world * 2 * W * k1p), dtype=torch.int32, device=dev)
        merged_val = torch.empty(W * k1p, dtype=torch.float32, device=dev)
        common = (Q, G, k1) + part + (W,)

        def strips():
            for i0, n in ((0, Q), (Q, G)):
                for c0 in range(0, n, W):
                    yield i0 + c0, min(W, n - c0)

        def contract(step, i0, wc):
            g_strip = None
            if i0 >= Q:                          # this rank's rows of the strip, zeros elsewhere, summed across the ranks
                c0 = i0 - Q
                lo, hi = max(c0, off), min(c0 + wc, off + self.G)
                raw[:wc].zero_()
                if lo < hi:
                    raw[lo - c0: hi - c0] = gf[lo - off: hi - off]
                words = (wc * D * raw.element_size() + 3) // 4
                dist_.all_reduce(raw.view(-1).view(torch.uint8)[: 4 * words].view(torch.int32), group=self.group)
                g_strip = PackedFeatures(raw[:wc], self.metric, self.normalize, self.precision, self.center)
            _lib.call("ieee_rerank_stream_part_contract", step, qpk.buf.data_ptr(), Q, _lib.ptr(gpart and gpart.buf),
                      _lib.ptr(g_strip and g_strip.buf), G, D, qpk.metric, qpk.precision, k1, *part, W, i0, wc,
                      colmax.data_ptr(), scratch.data_ptr(), sc_bytes, stream)

        for i0, wc in strips():                  # pass 0: colmax and rank
            contract(0, i0, wc)
            dist_.all_reduce(colmax[i0: i0 + wc].view(torch.int32), op=dist_.ReduceOp.MAX, group=self.group)
            n = 2 * wc * k1p
            mine, got = lists[:, :n], every[:, : world * n]
            _lib.call("ieee_rerank_stream_part_topk", *common, i0, wc, colmax.data_ptr(), mine[0].data_ptr(), mine[1].data_ptr(),
                      scratch.data_ptr(), sc_bytes, stream)
            for t in range(2):
                dist_.all_gather_into_tensor(got[t], mine[t].contiguous(), group=self.group)
            _lib.call("ieee_topk_merge", got[0].data_ptr(), got[1].data_ptr(), 2 * world, wc, k1p, rank[i0].data_ptr(),
                      merged_val.data_ptr(), stream)
        TRACE.mark("re-ranking: pass 0")
        # V's membership of every row from rank alone: no owned strips, so no gallery operand and no strip scratch
        _lib.call("ieee_rerank_stream_pass", 1, qpk.buf.data_ptr(), Q, None, G, D, qpk.metric, qpk.precision, k1, k2,
                  self.block_bytes, 0, 0, 0, 0, colmax.data_ptr(), rank.data_ptr(), ws.data_ptr(), ws.numel(), None, 0, stream)
        for i0, wc in strips():                  # pass 1: V's values
            contract(1, i0, wc)
            _lib.call("ieee_rerank_stream_part_members", *common[:3], k2, *common[3:], i0, wc, colmax.data_ptr(), ws.data_ptr(),
                      ws.numel(), scratch.data_ptr(), sc_bytes, stream)
            dist_.all_reduce(v_val[i0: i0 + wc], group=self.group)
            _lib.call("ieee_rerank_stream_part_weights", ws.data_ptr(), ws.numel(), Q, G, k1, k2, i0, wc, stream)
        TRACE.mark("re-ranking: pass 1")
        _lib.call("ieee_rerank_stream_finish", ws.data_ptr(), ws.numel(), Q, G, k1, k2, self.g_offset, self.G, rank.data_ptr(),
                  stream)

    def _gallery_range(self, ranges) -> PackedFeatures | None:
        """This rank's gallery range (rerank_ranges) packed with the evaluator's centre, or None when it is empty: the
        range's rows of the packed slice, then the rows up to the range's end, taken from the heads of the next slices
        (the rows before each one's own range, fewer than 256), all-gathered and packed here.  Packing is per row, so
        these are the bytes one GPU packs for these rows."""
        import torch.distributed as dist_
        gf, me, off, n = self._gallery_dev, dist_.get_rank(self.group), self.g_offset, self.G
        heads = [min(rows, a - o) for (o, rows, _), (a, _) in zip(self._slices, ranges)]
        h = max(heads)
        if h > 0:                                # the same verdict on every rank: all of them take part
            send = torch.zeros((h, gf.shape[1]), dtype=gf.dtype, device=self.device)
            send[: heads[me]] = gf[: heads[me]]
            recv = torch.empty((self.world, h, gf.shape[1]), dtype=gf.dtype, device=self.device)
            dist_.all_gather_into_tensor(recv.view(-1, gf.shape[1]), send, group=self.group)
        a, b = ranges[me]
        if a == b:
            return None
        slice_pk = self.chunks[0][1]
        if (a, b) == (off, off + n):
            return slice_pk
        pk = PackedFeatures._empty(b - a, slice_pk.D, self.metric, self.precision, self.center, self.device)
        _lib.call("ieee_packed_copy_rows", slice_pk.buf.data_ptr(), n, a - off, pk.buf.data_ptr(), b - a, 0, off + n - a,
                  pk.D, pk.precision, _lib.stream())
        if b > off + n:
            tail = torch.cat([recv[s, : heads[s]] for s in range(me + 1, self.world) if self._slices[s][0] < b])
            assert tail.shape[0] == b - (off + n)
            tpk = PackedFeatures(tail, self.metric, self.normalize, self.precision, self.center)
            _lib.call("ieee_packed_copy_rows", tpk.buf.data_ptr(), tail.shape[0], 0, pk.buf.data_ptr(), b - a, off + n - a,
                      tail.shape[0], pk.D, pk.precision, _lib.stream())
        return pk

    def _all_gather_owned(self, t: torch.Tensor, owned, Q: int, group=None):
        """Rows [q0, q1) and [Q + g0, Q + g1) of t ([Q + G, ...]), computed by each rank (owned = rerank_owned of every
        rank), from that rank into t on every rank of `group` (default: the gallery's): one all-gather, padded to the
        largest share."""
        import torch.distributed as dist_
        group = self.group if group is None else group
        dev = self.device
        idx = [torch.cat([torch.arange(q0, q1), torch.arange(Q + g0, Q + g1)]).to(dev) for q0, q1, g0, g1 in owned]
        rows = max(len(i) for i in idx)
        mine = idx[dist_.get_rank(group)]
        send = torch.zeros((rows,) + t.shape[1:], dtype=t.dtype, device=dev)
        send[: len(mine)] = t[mine]
        recv = torch.empty((len(owned) * rows,) + t.shape[1:], dtype=t.dtype, device=dev)
        dist_.all_gather_into_tensor(recv, send, group=group)
        at = torch.cat([r * rows + torch.arange(len(i), device=dev) for r, i in enumerate(idx)])
        t[torch.cat(idx)] = recv[at]

    def _gnn_prepare(self, qf: torch.Tensor, key):
        """GNN state of this query set: neighbours from row strips, the symbolic phase (one host round trip sizes every
        structure), then the numeric phase: A as CSR rows and the CSC of its gallery rows."""
        k1, k2 = self.k1, self.k2
        Q, D = qf.shape
        G = self.G
        N = Q + G
        if k1 > N:
            raise ValueError('rerank="gnn": k1 = {} exceeds the {} query and gallery samples'.format(k1, N))
        lib = _lib.load()
        sc_bytes = lib.ieee_gnn_stream_scratch_bytes(Q, G, k1, self.block_bytes)
        if sc_bytes == 0:
            raise ValueError('rerank="gnn": ' + lib.ieee_last_error().decode())
        qpk = self._take_early_q(qf)
        if qpk is None:
            qpk = PackedFeatures(qf, self.metric, self.normalize, self.precision, None)
        gpk = self.chunks[0][1]
        dev = self.device
        scratch = torch.empty(sc_bytes, dtype=torch.uint8, device=dev)     # strips, then the graph calls' index
        rank = torch.empty((N, k1), dtype=torch.int32, device=dev)
        S = torch.empty((N, k1), dtype=torch.float32, device=dev)
        if self.query_group is not None:
            state = self._gnn_prepare_shared(qpk, gpk, rank, S, scratch)
            return dict(state, key=key, qf=qf, Q=Q, k1=k1, k2=k2, rank=rank, S=S, scratch_bytes=sc_bytes)
        _lib.call("ieee_gnn_stream_neighbours", qpk.buf.data_ptr(), Q, gpk.buf.data_ptr(), G, D, qpk.precision, k1,
                  self.block_bytes, rank.data_ptr(), S.data_ptr(), scratch.data_ptr(), sc_bytes, _lib.stream())
        TRACE.mark("GNN neighbours")
        sizes = (C.c_int64 * 6)()
        _lib.call("ieee_gnn_stream_graph_bytes_sync", rank.data_ptr(), Q, G, k1, k2, scratch.data_ptr(), sc_bytes, sizes,
                  _lib.stream())
        TRACE.mark("GNN symbolic phase")
        nnz, nnz_g, work_bytes = sizes[0], sizes[1], sizes[2]
        work = torch.empty(work_bytes, dtype=torch.uint8, device=dev)    # released (stream-ordered) on return
        a_ptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
        a_col = torch.empty(nnz, dtype=torch.int32, device=dev)
        a_val = torch.empty(nnz, dtype=torch.float32, device=dev)
        g_ptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
        g_row = torch.empty(nnz_g, dtype=torch.int32, device=dev)
        g_val = torch.empty(nnz_g, dtype=torch.float32, device=dev)
        _lib.call("ieee_gnn_stream_graph", rank.data_ptr(), S.data_ptr(), Q, G, k1, k2, scratch.data_ptr(), sc_bytes,
                  work.data_ptr(), work_bytes, sizes, a_ptr.data_ptr(), a_col.data_ptr(), a_val.data_ptr(), g_ptr.data_ptr(),
                  g_row.data_ptr(), g_val.data_ptr(), _lib.stream())
        TRACE.mark("GNN numeric phase")
        return {"key": key, "qf": qf, "Q": Q, "k1": k1, "k2": k2, "rank": rank, "S": S, "a_ptr": a_ptr, "a_col": a_col,
                "a_val": a_val, "g_ptr": g_ptr, "g_row": g_row, "g_val": g_val, "scratch_bytes": sc_bytes,
                "work_bytes": work_bytes}

    def _gnn_prepare_shared(self, qpk: PackedFeatures, gpk: PackedFeatures, rank, S, scratch):
        """_gnn_prepare's calls in phases, shared by the ranks of query_group (all holding the whole gallery and query set):
        each rank computes the rows it owns (rerank_owned) of every stage whose work grows as N^2, and replicates the
        stages linear in the adjacency's entries.  Neighbour lists and counts are all-gathered; the CSR structures and
        the CSC, where every rank holds zeros but in its own rows, are summed as int32 (an exact move of each entry's bits).
        Every rank ends with the one-GPU rank, S, a_ptr, A's gallery rows and CSC, and its own query rows of A."""
        import torch.distributed as dist_
        qg = self.query_group
        Q, G, k1, k2 = qpk.rows, self.G, self.k1, self.k2
        N, dev, stream = Q + G, self.device, _lib.stream()
        owned = [rerank_owned(Q, G, self._q_world, r) for r in range(self._q_world)]
        own = owned[self._q_rank]
        sc = (scratch.data_ptr(), scratch.numel())

        def summed(t):
            dist_.all_reduce(t.view(torch.int32), group=qg)

        _lib.call("ieee_gnn_stream_neighbours_rows", qpk.buf.data_ptr(), Q, gpk.buf.data_ptr(), G, qpk.D, qpk.precision, k1,
                  self.block_bytes, *own, rank.data_ptr(), S.data_ptr(), *sc, stream)
        TRACE.mark("GNN neighbours")
        for t in (rank, S):
            self._all_gather_owned(t, owned, Q, qg)
        TRACE.mark("GNN exchange: rank, S")
        _lib.call("ieee_gnn_stream_symbolic", rank.data_ptr(), Q, G, k1, k2, *own, *sc, stream)
        TRACE.mark("GNN symbolic phase")
        off = (C.c_size_t * 10)()
        _lib.call("ieee_gnn_stream_layout", Q, G, k1, k2, None, off)
        if k2 != 1:
            for i in range(4):
                self._all_gather_owned(scratch[off[i]: off[i] + 4 * N].view(torch.int32), owned, Q, qg)
        TRACE.mark("GNN exchange: counts")
        sizes = (C.c_int64 * 6)()
        _lib.call("ieee_gnn_stream_sizes_sync", Q, G, k1, k2, *sc, sizes, stream)
        TRACE.mark("GNN sizes")
        nnz, nnz_g, work_bytes = sizes[0], sizes[1], sizes[2]
        work = torch.empty(work_bytes, dtype=torch.uint8, device=dev)    # released (stream-ordered) on return
        a_ptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
        a_col = torch.empty(nnz, dtype=torch.int32, device=dev)
        a_val = torch.empty(nnz, dtype=torch.float32, device=dev)
        g_ptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
        g_row = torch.empty(nnz_g, dtype=torch.int32, device=dev)
        g_val = torch.empty(nnz_g, dtype=torch.float32, device=dev)
        a = (a_ptr.data_ptr(), a_col.data_ptr(), a_val.data_ptr())

        def numeric(step):
            _lib.call("ieee_gnn_stream_numeric", step, rank.data_ptr(), S.data_ptr(), Q, G, k1, k2, *own, *sc, work.data_ptr(),
                      work_bytes, sizes, *a, stream)
            TRACE.mark("GNN numeric step %d" % step)

        if k2 != 1:
            _lib.call("ieee_gnn_stream_layout", Q, G, k1, k2, sizes, off)
            for step, n in enumerate((sizes[3], sizes[4], sizes[5])):        # B1, A1, B2: columns and values
                numeric(step)
                for o in (off[4 + 2 * step], off[5 + 2 * step]):
                    summed(work[o: o + 4 * n])
                TRACE.mark("GNN exchange after step %d" % step)
        numeric(3)
        summed(a_col[nnz - nnz_g:])                     # A2's gallery rows: its query rows stay with their owners
        summed(a_val[nnz - nnz_g:])
        TRACE.mark("GNN exchange: gallery rows of A")
        _lib.call("ieee_gnn_stream_csc", Q, G, k1, *own, *sc, *a, g_ptr.data_ptr(), g_row.data_ptr(), g_val.data_ptr(), stream)
        TRACE.mark("GNN CSC")
        summed(g_row)
        summed(g_val)
        TRACE.mark("GNN exchange: CSC")
        return {"a_ptr": a_ptr, "a_col": a_col, "a_val": a_val, "g_ptr": g_ptr, "g_row": g_row, "g_val": g_val,
                "work_bytes": work_bytes}

    def _gnn_block(self, s: int, e: int) -> torch.Tensor:
        """-(A[q] . A[Q + g]) of queries [s, e) into the scratch block (accumulated in float64): no contraction."""
        dist = self._block[: e - s]
        if e > s:
            rr = self._rr
            if self._rr_scratch is None or self._rr_scratch.numel() < (e - s) * self.G:
                self._rr_scratch = torch.empty((e - s) * self.G, dtype=torch.float64, device=self.device)
            _lib.call("ieee_gnn_stream_block", rr["a_ptr"].data_ptr(), rr["a_col"].data_ptr(), rr["a_val"].data_ptr(),
                      rr["g_ptr"].data_ptr(), rr["g_row"].data_ptr(), rr["g_val"].data_ptr(), rr["Q"], self.G, s, e - s,
                      dist.data_ptr(), dist.stride(0), self._rr_scratch.data_ptr(), 8 * self._rr_scratch.numel(),
                      _lib.stream())
            TRACE.mark("  GNN similarity")
        return dist

    def _rerank_block(self, dist: torch.Tensor, row0: int) -> torch.Tensor:
        """Queries [row0, row0 + rows) of the prepared set: distances to this rank's gallery rows -> re-ranked distances,
        in place."""
        rr = self._rr
        rows = dist.shape[0]
        if rows == 0:                            # (an empty query set has no state to blend with)
            return dist
        if self._rr_scratch is None or self._rr_scratch.numel() < rows * self.G:
            self._rr_scratch = torch.empty(rows * self.G, dtype=torch.float32, device=self.device)
        _lib.call("ieee_rerank_stream_block_window", rr["ws"].data_ptr(), rr["Q"], self.g_total, rr["k1"], rr["k2"], self.G,
                  rr["colmax"].data_ptr(), row0, rows, self.lambda_value, dist.data_ptr(), dist.stride(0),
                  self._rr_scratch.data_ptr(), 4 * self._rr_scratch.numel(), _lib.stream())
        TRACE.mark("  re-ranking blend")
        return dist

    def _prepare_gallery(self, qf_dev):
        """ieee_gallery_prepare: grouping + [centre from the query rows] + packing of a device-resident gallery -- and
        of the query rows themselves when they make one block: the host work between this call and the evaluation call
        then hides behind that kernel (a small gallery shard alone is packed before the next call arrives).  The
        grouping stays on the library's side stream until a consumer joins it (GalleryLabels.wait)."""
        gf = self._gallery_dev
        if gf.stride(1) != 1:
            gf = self._gallery_dev = gf.contiguous()
        G, D = gf.shape
        src, ws, qpk, flags = None, None, None, _lib.PREPARE_DEFER_JOIN
        if qf_dev is not None and qf_dev.shape[0] > 0:
            src = qf_dev if qf_dev.stride(1) == 1 else qf_dev.contiguous()
            assert src.dtype == gf.dtype, "query and gallery features must have the same dtype"
        if src is not None and self._use_center and self.center is None:
            self.center = torch.empty(D, dtype=torch.float32, device=self.device)
        else:
            flags |= _lib.PREPARE_KEEP_CENTER
        center = self.center if self._use_center else None
        pk = PackedFeatures._empty(G, D, self.metric, self.precision, center, self.device)
        if src is not None and src.shape[0] <= self._block_rows_for(src.shape[0], G):
            qpk = PackedFeatures._empty(src.shape[0], D, self.metric, self.precision, center, self.device)
            self._early_q = (_features_key(qf_dev), qpk)
        cur = torch.cuda.current_stream()
        _lib.call("ieee_gallery_prepare", gf.data_ptr(), gf.stride(0), _lib.DTYPES[gf.dtype], G, D, pk.metric, int(self.normalize),
                  pk.precision, self.labels.pids.data_ptr(), _lib.ptr(src), src.stride(0) if src is not None else 0,
                  src.shape[0] if src is not None else 0, _lib.ptr(center), pk.buf.data_ptr(),
                  self.labels.group.data_ptr(), qpk.buf.data_ptr() if qpk is not None else None, flags, _lib.ptr(ws),
                  cur.cuda_stream)
        self.labels.ready = cur.record_event()
        self.labels.side_join = True
        self.chunks = [(0, pk)]

    def _take_early_q(self, qf: torch.Tensor):
        """The packed form of exactly these query rows, if _prepare_gallery made it (used once)."""
        early, self._early_q = self._early_q, None
        if early is not None and early[0] == _features_key(qf):
            return early[1]
        return None

    def _ensure_center(self, qf_dev: torch.Tensor):
        """Fix the centre (first query set seen) and prepare a device-resident gallery with it."""
        if self._gallery_dev is not None and not self.chunks:
            self._prepare_gallery(qf_dev)
        elif self._use_center and self.center is None:
            self.center = feature_center(qf_dev, self.normalize)

    # -- one query block ---------------------------------------------------------------------------------
    def _block_rows_for(self, Q: int, G: int) -> int:
        # re-ranking: the distance block and its accumulators share the budget (k-reciprocal: float32, as large as the
        # block; GNN: float64, twice as large)
        budget = self.block_bytes // (3 if self.gnn else 2) if self.rerank else self.block_bytes
        rows = max(128, int(budget // (4 * max(G, 1))) // 128 * 128)
        return min(Q, rows)

    def _block_rows(self, Q: int) -> int:
        return self._block_rows_for(Q, self.G)

    def _ensure_block(self, rows: int):
        if self._block is None or self._block.shape[0] < rows:
            self._block = self._new_block(rows)

    def _new_block(self, rows: int) -> torch.Tensor:
        # row pitch padded to 128 bytes: the contraction's TMA-store epilogue and the rank kernels'
        # 16-byte loads both want aligned rows (G itself is arbitrary, e.g. 15913)
        pitch = (self.G + 31) // 32 * 32
        return torch.empty((rows, pitch), dtype=torch.float32, device=self.device)[:, : self.G]

    def _distance_block(self, qpk: PackedFeatures) -> torch.Tensor:
        """Distances of one packed query block against this rank's gallery rows, into the scratch block."""
        out = self._block[: qpk.rows]
        for i, (c0, gpk) in enumerate(self.chunks):
            if isinstance(gpk, tuple):            # (event, host->device staging tensor): pack on arrival
                ev, staged = gpk
                torch.cuda.current_stream().wait_event(ev)
                gpk = PackedFeatures(staged, self.metric, self.normalize, self.precision, self.center)
                self.chunks[i] = (c0, gpk)        # packed once, reused by later query blocks
            packed_distmat(qpk, gpk, out[:, c0: c0 + gpk.rows])
            TRACE.mark("  chunk %d contraction" % c0)
        return out

    def _query_blocks(self, qf: torch.Tensor, rows: int, pack0: PackedFeatures | None = None, q_event=None):
        """Iterates over (s, e, distances of queries [s, e)) in blocks of `rows`: each block is packed (block 0 may come
        packed as `pack0`), after `q_event` when the queries are still being copied, contracted against every gallery
        chunk and, on a re-ranking evaluator, re-ranked.  Block 0 is queued before this returns, so the caller can hide
        host work behind its contraction; every later block when the iteration reaches it, in the same scratch.  With a
        query_group only this rank's queries (_query_range) are iterated."""
        q0, Q = self._query_range(qf.shape[0])
        self._ensure_block(rows)

        def block(s, e, qpk):
            if self.gnn:
                return self._gnn_block(s, e)
            if qpk is None:
                if q_event is not None:
                    torch.cuda.current_stream().wait_event(q_event)
                qpk = PackedFeatures(qf[s:e], self.metric, self.normalize, self.precision, self.center)
            dist = self._distance_block(qpk)
            return self._rerank_block(dist, s) if self.rerank else dist

        dist0 = block(q0, min(Q, q0 + rows), pack0)

        def blocks():
            for s in range(q0, Q, rows):
                e = min(Q, s + rows)
                yield s, e, dist0 if s == q0 else block(s, e, None)
        return blocks()

    def _copy_stream(self) -> torch.cuda.Stream:
        """The copy stream, ordered after the work queued on the compute stream so far."""
        if self._copy is None:
            self._copy = copy_stream(self.device)
        self._copy.wait_stream(torch.cuda.current_stream())
        return self._copy

    def ranked_lists(self, qf: torch.Tensor, q_pids=None, q_camids=None, k: int = 10):
        """First ``k`` entries of every query's junk-filtered ranked list over the WHOLE (possibly sharded) gallery --
        what ``visualize_ranked_results`` walks (torchreid/utils/reidtools.py:49,109-145).

        Each rank selects the k best kept items of its gallery slice (``ieee_topk`` with global indices), the
        per-shard lists are all-gathered and merged (``ieee_topk_merge``): k * world candidates per query instead of
        a Q x G matrix on one device.  Ties go to the lower global gallery index, as on one GPU.  Pass no labels for an
        unmasked top-k.  Returns (idx int32 [Q, k'] global gallery indices, -1 padded; dist float32 [Q, k']) on the
        device, identical on every rank; k' = min(k, total gallery size)."""
        qf = _as_features(qf)
        masked = q_pids is not None
        with torch.cuda.device(self.device):
            qf = qf.to(self.device, non_blocking=True)
            Q = qf.shape[0]
            if self.query_group is not None:
                self._agree_on_queries(qf)
            k_eff = max(1, min(int(k), self.g_total))
            idx = torch.empty((Q, k_eff), dtype=torch.int32, device=self.device)
            val = torch.empty((Q, k_eff), dtype=torch.float32, device=self.device)
            if Q == 0:
                return idx, val
            self._ensure_center(qf)
            if self.rerank:
                self._rerank_prepare(qf)
            self._early_q = None          # (this path packs its query blocks itself: do not keep the early copy alive)
            if self._host_gallery is not None:
                self._start_gallery_copies(self._copy_stream())
            qp = _as_device(q_pids, torch.int64, self.device) if masked else None
            qc = _as_device(q_camids, torch.int64, self.device) if masked else None
            self.labels.wait(torch.cuda.current_stream())
            for s, e, dist in self._query_blocks(qf, self._block_rows(Q)):
                loc_i = idx[s:e] if self.world == 1 else torch.empty((e - s, k_eff), dtype=torch.int32, device=self.device)
                loc_v = val[s:e] if self.world == 1 else torch.empty((e - s, k_eff), dtype=torch.float32, device=self.device)
                _lib.call("ieee_topk", dist.data_ptr(), dist.stride(0), e - s, self.G, self.g_offset,
                          _lib.ptr(qp[s:e] if masked else None), _lib.ptr(qc[s:e] if masked else None),
                          self.labels.pids.data_ptr() if masked else None, self.labels.camids.data_ptr() if masked else None,
                          k_eff, loc_i.data_ptr(), loc_v.data_ptr(), _lib.stream())
                if self.world > 1:
                    import torch.distributed as dist_
                    all_i = torch.empty((self.world, e - s, k_eff), dtype=torch.int32, device=self.device)
                    all_v = torch.empty((self.world, e - s, k_eff), dtype=torch.float32, device=self.device)
                    dist_.all_gather_into_tensor(all_i, loc_i, group=self.group)
                    dist_.all_gather_into_tensor(all_v, loc_v, group=self.group)
                    _lib.call("ieee_topk_merge", all_i.data_ptr(), all_v.data_ptr(), self.world, e - s, k_eff,
                              idx[s:e].data_ptr(), val[s:e].data_ptr(), _lib.stream())
            if self.query_group is not None:
                for t in (idx, val):
                    self._all_gather_owned(t, self._owned_queries(Q), Q, self.query_group)
        return idx, val

    def _owned_queries(self, Q: int):
        """The query rows every rank of query_group evaluates, in _all_gather_owned's form."""
        return [rerank_owned(Q, self.G, self._q_world, r)[:2] + (0, 0) for r in range(self._q_world)]

    def _rank_block_peer(self, dist, qp, qc, link, Qb_max, Qtot, q_base, cap, W, stats, cmc, summ, stats_out, k_eff):
        """gather -> count -> metrics of one query block with the exchanges as stores into peer memory; the metrics
        kernel of the last block also reduces over all queries."""
        Qb = dist.shape[0]
        ex = link.descriptor(Qb_max, Qb, Qtot, q_base, cap, W, link.next_epoch())
        junk = torch.empty((Qb, cap), dtype=torch.int64, device=self.device)
        n_rel = torch.empty(Qb, dtype=torch.int32, device=self.device)
        n_junk = torch.empty(Qb, dtype=torch.int32, device=self.device)
        cur = torch.cuda.current_stream()
        self.labels.wait(cur)
        st = cur.cuda_stream
        _lib.call("ieee_rank_gather_peer", dist.data_ptr(), dist.stride(0), self.G, qp.data_ptr(), qc.data_ptr(),
                  self.labels.camids.data_ptr(), self.labels.group.data_ptr(), self.g_offset, n_rel.data_ptr(), junk.data_ptr(),
                  n_junk.data_ptr(), stats.data_ptr(), C.byref(ex), st)
        TRACE.mark("  gather (lists stored into every peer)")
        _lib.call("ieee_rank_count_peer", dist.data_ptr(), dist.stride(0), self.G, self.g_offset, n_rel.data_ptr(),
                  junk.data_ptr(), n_junk.data_ptr(), stats.data_ptr(), C.byref(ex), st)
        TRACE.mark("  count (partial counts stored into every peer)")
        _lib.call("ieee_rank_metrics_peer", self.g_total, k_eff, stats.data_ptr(), cmc.data_ptr(), summ.data_ptr(),
                  stats_out.data_ptr(), C.byref(ex), st)
        TRACE.mark("  metrics (+ reduction on the last block)")
        return ex

    def _rank_block(self, dist, qp, qc, cap, width, ap, first, short, ties, inp):
        Qb = dist.shape[0]
        st = _stages_for(Qb, cap, self.world, self.device, width)
        self.labels.wait(torch.cuda.current_stream())
        st.gather(dist, qp, qc, self.labels, self.g_offset, stats=ties)     # kernels max / add straight into `ties`
        TRACE.mark("  gather")
        if self.world > 1:
            import torch.distributed as dist_
            # the lists carry their own lengths (last column): one all-gather, then one all-reduce of the counts
            rel_all = torch.empty((self.world, Qb, cap + 1), dtype=torch.int64, device=self.device)
            dist_.all_gather_into_tensor(rel_all, st.rel, group=self.group)
            TRACE.mark("  all-gather of relevant lists")
            st.count(dist, self.G, self.g_offset, rel_all)
            TRACE.mark("  count")
            dist_.all_reduce(st.counts, group=self.group)
            TRACE.mark("  all-reduce of counts")
        else:
            st.count(dist, self.G, self.g_offset)
        _lib.call("ieee_rank_query_metrics", st.counts.data_ptr(), Qb, self.g_total, 1, st.width, self.max_rank,
                  ap.data_ptr(), first.data_ptr(), short.data_ptr(), inp.data_ptr(), _lib.stream())
        TRACE.mark("  query metrics")
        return st

    @classmethod
    def from_host(cls, gf_host: torch.Tensor, g_pids, g_camids, dist_metric="euclidean", normalize_feature=False,
                  precision=None, max_rank=20, num_chunks=8, device=None, **kw):
        """Gallery features in (pinned) host memory: the copy is split into row chunks on a copy stream; each chunk is
        packed and multiplied as soon as it lands, so PCIe time and tensor-core time overlap."""
        _lib.require_cuda()
        dev = device or torch.device("cuda", torch.cuda.current_device())
        gf_host = _as_features(gf_host)
        with torch.cuda.device(dev):
            self = cls(None, g_pids, g_camids, dist_metric, normalize_feature,
                       precision or ("bf16" if gf_host.dtype == torch.bfloat16 else "f16x3"), max_rank, **kw)
        assert gf_host.shape[0] == self.G
        self._host_gallery, self._num_chunks = gf_host, num_chunks      # copies start in evaluate(), after the queries'
        return self

    def _start_gallery_copies(self, copy: torch.cuda.Stream):
        gf_host, G = self._host_gallery, self.G
        step = max(256, ((G + self._num_chunks - 1) // self._num_chunks + 255) // 256 * 256)   # whole 256-column tiles
        for c0 in range(0, G, step):
            c1 = min(G, c0 + step)
            staged = torch.empty((c1 - c0, gf_host.shape[1]), dtype=gf_host.dtype, device=self.device)
            with torch.cuda.stream(copy):
                staged.copy_(gf_host[c0:c1], non_blocking=True)
                ev = copy.record_event()
            self.chunks.append((c0, (ev, staged)))
        self._host_gallery = None

    def _memo_key(self, q_pids):
        """Key of these labels in the capacity memo; None when a label set is not a torch tensor (no identity to key on)."""
        if self._label_keys[0] is None or _tensor_key(q_pids) is None:
            return None
        return (self._label_keys, _tensor_key(q_pids), self.world)

    def _one_resident_block(self, qf: torch.Tensor) -> bool:
        """Queries in HBM that make one block against a gallery packed in HBM as one chunk: what a one-call evaluation
        takes."""
        return (qf.is_cuda and self._host_gallery is None and len(self.chunks) == 1
                and isinstance(self.chunks[0][1], PackedFeatures) and 0 < qf.shape[0] <= self._block_rows(qf.shape[0]))

    def _evaluate_one_call(self, qf, q_pids, q_camids, return_distmat, memo_key, cap, width):
        """One resident block: the whole evaluation is ONE foreign call, which enqueues pack -> contraction -> gather ->
        count -> metrics -> reduce back to back from C, and one device->host copy of the result block.  On one GPU that
        is ieee_retrieve_eval_prepared (cap <= 0: size the lists here first).  A sharded gallery takes
        ieee_retrieve_eval_prepared_peer with the sizes an earlier evaluation with the same labels memoised: no
        collective launch, no host round trip before the result."""
        peer = self.world > 1
        with torch.cuda.device(self.device):
            lib = _lib.load()
            Q, D = qf.shape
            if qf.stride(1) != 1:
                qf = qf.contiguous()
            qp = _as_device(q_pids, torch.int64, self.device)
            qc = _as_device(q_camids, torch.int64, self.device)
            k_eff = min(self.max_rank, self.g_total)
            prec = _lib.PRECISIONS[self.precision]
            cur = torch.cuda.current_stream()
            if peer:
                entry, W = "ieee_retrieve_eval_prepared_peer", min(width, self.world * cap)
                link = link_for(self.group, self.device, lib.ieee_peer_exchange_bytes(Q, Q, cap, W, self.world))
                ex = link.descriptor(Q, Q, Q, 0, cap, W, link.next_epoch())
                ws_bytes = lib.ieee_retrieve_prepared_peer_workspace_bytes(Q, D, prec, cap)
            else:
                entry, W = "ieee_retrieve_eval_prepared", 0          # (no merged lists on one GPU)
                if cap <= 0:
                    # sizing pass: the capacity query synchronises once; later calls with the same labels skip it
                    cap = self.labels.list_cap(qp)
                    if memo_key is not None:
                        _memo_put(memo_key, (cap, 0), (self._label_refs, q_pids))
                ws_bytes = lib.ieee_retrieve_prepared_workspace_bytes(Q, D, prec, cap)
            ws, res = _one_call_buffers((entry, Q, D, prec, cap, k_eff, str(self.device)), ws_bytes, 96 + 4 * k_eff, self.device)
            self._ensure_block(Q)
            # per-query results straight into fresh arrays (with the peer exchange every rank derives all of them
            # itself): nothing to copy out after the result has arrived, when the GPU would be idle
            ap = torch.empty(Q, dtype=torch.float64, device=self.device)
            first = torch.empty(Q, dtype=torch.int32, device=self.device)
            self.labels.wait(cur, join=False)
            qpk = self._take_early_q(qf)          # packed already by ieee_gallery_prepare (first evaluation of this gallery)
            self._one_call_launch(qf, qp, qc, cap, self._block, ws, res, ap, first, qpk, ex if peer else None)
            (overflow, longest), summary, cmc = _read_result(res)
        if overflow or longest > W:
            return self._retry(qf, q_pids, q_camids, return_distmat, memo_key, cap, longest, one_call=True)
        return self._result(summary, cmc, cap, ap, first, self._block[:Q].clone() if return_distmat else None)

    def _one_call_launch(self, qf, qp, qc, cap, block, ws, res, ap, first, qpk=None, ex=None, epoch=None):
        """Enqueue one resident block's evaluation on the current stream: ieee_retrieve_eval_prepared (cap > 0 here, or
        <= 0 to size the lists first), or with an exchange descriptor `ex` ieee_retrieve_eval_prepared_peer, whose epoch
        comes from `ex` or, with `epoch` (int64 [1] on the device), from that word (..._dev_epoch).  Results go into
        `res` (the result block), `ap`, `first` and the distance block `block`."""
        Q, D = qf.shape
        queries = (qf.data_ptr(), qf.stride(0), _lib.DTYPES[qf.dtype], Q, D, _lib.METRICS[self.metric], int(self.normalize),
                   _lib.PRECISIONS[self.precision], self.chunks[0][1].buf.data_ptr(), self.labels.group.data_ptr(),
                   _lib.ptr(self.center), self.G)
        rest = (qpk.buf.data_ptr() if qpk is not None else None, ws.data_ptr(), ws.numel(), _lib.stream())
        outs = (block.data_ptr(), block.stride(0), res.data_ptr() + 96, res.data_ptr() + 32)
        if ex is None:
            _lib.call("ieee_retrieve_eval_prepared", *queries, qp.data_ptr(), qc.data_ptr(), self.labels.camids.data_ptr(),
                      self.max_rank, cap, None, *outs, ap.data_ptr(), first.data_ptr(), *rest)
        elif epoch is None:
            _lib.call("ieee_retrieve_eval_prepared_peer", *queries, self.g_total, self.g_offset, qp.data_ptr(), qc.data_ptr(),
                      self.labels.camids.data_ptr(), self.max_rank, *outs, res.data_ptr(), ap.data_ptr(), first.data_ptr(),
                      C.byref(ex), *rest)
        else:
            _lib.call("ieee_retrieve_eval_prepared_peer_dev_epoch", *queries, self.g_total, self.g_offset, qp.data_ptr(),
                      qc.data_ptr(), self.labels.camids.data_ptr(), self.max_rank, *outs, res.data_ptr(), ap.data_ptr(),
                      first.data_ptr(), C.byref(ex), epoch.data_ptr(), *rest)

    def _evaluate_staged(self, qf, q_pids, q_camids, return_distmat, memo_key, cap, width):
        """The query-block loop, stage by stage: any number of blocks, host queries and a host gallery, re-ranking, and
        both exchanges of a sharded gallery.  cap <= 0: the capacity is queried behind block 0's contraction."""
        import torch.distributed as dist_
        with torch.cuda.device(self.device):
            TRACE.mark("evaluate: start")
            Q = qf.shape[0]
            rows = self._block_rows(Q)
            # queries already in HBM: pack the first block before anything else, so the GPU is busy while the host
            # prepares the rest of the step
            early_pack = None
            if self.rerank and Q > 0:
                rr = self._rerank_prepare(qf)
                early_pack = rr.get("packed") if rows >= Q else None
            if qf.is_cuda and early_pack is None and not self.gnn:
                early_pack = self._take_early_q(qf) if rows >= Q else None
                if early_pack is None:
                    early_pack = PackedFeatures(qf[: min(Q, rows)], self.metric, self.normalize, self.precision, self.center)
            # small label copies go FIRST: host->device transfers of every stream share one copy engine queue, so a
            # label copy issued after the feature copies would hold the compute stream until they have all landed
            qp = _as_device(q_pids, torch.int64, self.device)
            qc = _as_device(q_camids, torch.int64, self.device)
            ids_ready = torch.cuda.current_stream().record_event()
            q_event = None
            if not qf.is_cuda or self._host_gallery is not None:
                copy = self._copy_stream()
                if not qf.is_cuda:                       # queries first: every contraction needs them
                    if self.world > 1:
                        # the query set is the same on every rank: each copies 1/N of it over its own PCIe link and
                        # the slices are all-gathered over NVLink instead of N full host->device copies
                        rank = dist_.get_rank(self.group)
                        per = (Q + self.world - 1) // self.world
                        q_all = torch.empty((self.world * per, qf.shape[1]), dtype=qf.dtype, device=self.device)
                        mine = q_all[rank * per: (rank + 1) * per]
                        lo, hi = min(Q, rank * per), min(Q, (rank + 1) * per)
                        with torch.cuda.stream(copy):
                            if hi > lo:
                                mine[: hi - lo].copy_(qf[lo:hi], non_blocking=True)
                            if hi - lo < per:
                                mine[hi - lo:].zero_()
                            dist_.all_gather_into_tensor(q_all, mine, group=self.group)
                            q_event = copy.record_event()
                        qf = q_all[:Q]
                    else:
                        q_dev = torch.empty(qf.shape, dtype=qf.dtype, device=self.device)
                        with torch.cuda.stream(copy):
                            q_dev.copy_(qf, non_blocking=True)
                            q_event = copy.record_event()
                        qf = q_dev
                if self._host_gallery is not None:
                    self._start_gallery_copies(copy)
                if q_event is not None and Q > 0:
                    # host queries: the centre comes from their device copy, before any chunk is packed
                    torch.cuda.current_stream().wait_event(q_event)
                    self._ensure_center(qf)
            ap = torch.empty(Q, dtype=torch.float64, device=self.device)
            first = torch.empty(Q, dtype=torch.int32, device=self.device)
            short = torch.empty(Q, dtype=torch.int32, device=self.device)
            inp = torch.empty(Q, dtype=torch.float64, device=self.device)
            k_eff = min(self.max_rank, self.g_total)
            res = torch.zeros(96 + 4 * k_eff, dtype=torch.uint8, device=self.device)    # the kernels accumulate into it
            ties, summ, cmc = res[:32].view(torch.int64), res[32:96], res[96:].view(torch.float32)
            blocks = self._query_blocks(qf, rows, early_pack, q_event)
            TRACE.mark("contraction(block 0) queued")
            if cap <= 0:
                # The contraction of the first block is queued FIRST; the capacity is then queried on a side stream
                # that only waits for the gallery grouping and the query ids, so its host round trip (and the
                # host-side allocations below) hide behind the tensor-core kernel.
                cap_done, cap_host = self.labels.list_cap_async(qp, ids_ready)
                cap_done.synchronize()
                cap = max(int(cap_host.item()), 1)
                if self.world > 1:
                    # every rank must size its lists alike for the all-gather (after the contraction: a NCCL kernel
                    # beside the persistent GEMM would take an SM pair away from a tile cluster)
                    cap_t = torch.tensor([cap], dtype=torch.int32, device=self.device)
                    dist_.all_reduce(cap_t, op=dist_.ReduceOp.MAX, group=self.group)
                    cap = int(cap_t.item())
            W = min(width, self.world * cap) if width > 0 else self.world * cap     # row width of the merged counts
            peer = self.world > 1 and self.exchange == "peer" and Q > 0
            q0, q1 = self._query_range(Q)
            full = torch.empty((q1 - q0, self.G), dtype=torch.float32, device=self.device) if return_distmat else None
            if peer:
                lib = _lib.load()
                link = link_for(self.group, self.device, lib.ieee_peer_exchange_bytes(rows, Q, cap, W, self.world))
                stats = torch.zeros(4, dtype=torch.int64, device=self.device)      # this rank's own statistics
            for s, e, dist in blocks:
                if peer:
                    self._rank_block_peer(dist, qp[s:e], qc[s:e], link, rows, Q, s, cap, W, stats, cmc, summ, ties, k_eff)
                else:
                    self._rank_block(dist, qp[s:e], qc[s:e], cap, width, ap[s:e], first[s:e], short[s:e], ties, inp[s:e])
                if full is not None:
                    full[s - q0:e - q0].copy_(dist)
            if not peer and self.world > 1:
                dist_.all_reduce(ties[:2], group=self.group)          # [2] (longest merged list) is the same on every rank
            if self.query_group is not None:
                # every rank's per-query results in query order, and the statistics of all queries: the reduction below
                # then runs on the same inputs on every rank, and a list overflow is decided by all of them together
                for t in (ap, first, short, inp):
                    self._all_gather_owned(t, self._owned_queries(Q), Q, self.query_group)
                dist_.all_reduce(ties[:2], group=self.query_group)
                dist_.all_reduce(ties[2:3], op=dist_.ReduceOp.MAX, group=self.query_group)
            TRACE.mark("rank stages done")
            if peer:
                offs = [lib.ieee_peer_result_offset(i, rows, Q, cap, W, self.world) for i in (0, 1)]
                ap = link.view[offs[0]: offs[0] + 8 * Q].view(torch.float64)       # every rank holds all per-query results
                first = link.view[offs[1]: offs[1] + 4 * Q].view(torch.int32)
            else:
                _lib.call("ieee_rank_reduce", ap.data_ptr(), first.data_ptr(), short.data_ptr(), Q, k_eff, ties.data_ptr() + 8,
                          cmc.data_ptr(), summ.data_ptr(), inp.data_ptr(), _lib.stream())
            TRACE.mark("reduce done")
            (overflow, longest), summary, cmc_host = _read_result(res)
            if peer:
                ap, first = ap.clone(), first.clone()    # the exchange buffer is overwritten by the next evaluation
        if overflow or longest > W:
            return self._retry(qf, q_pids, q_camids, return_distmat, memo_key, cap, longest, one_call=False)
        if memo_key is not None:
            _memo_put(memo_key, (cap, max(longest, 1)), (self._label_refs, q_pids))
        TRACE.report()
        return self._result(summary, cmc_host, cap, ap, first, full)

    def _retry(self, qf, q_pids, q_camids, return_distmat, memo_key, cap, longest, one_call):
        """A list did not fit the sizes the capacity memo held: forget them and evaluate again with exact ones.  The
        one-GPU one-call route sizes exactly itself (and memoises the new capacity); every other route runs the
        staged loop without the memo.  Exact sizes cannot overflow, so an overflow with them is an error."""
        if memo_key is None:
            raise RuntimeError("ieee_b200: per-query lists overflowed an exactly sized buffer (cap=%d, longest=%d)" % (cap, longest))
        _memo_drop(memo_key)
        if one_call and self.world == 1:
            return self._evaluate_one_call(qf, q_pids, q_camids, return_distmat, memo_key, 0, 0)
        return self.evaluate(qf, q_pids, q_camids, return_distmat, use_cap_memo=False, one_call=False)

    def _result(self, summary, cmc, cap, ap, first, distmat):
        raise_for_status(summary, self.max_rank)
        info = {"num_valid": summary.num_valid, "num_ties": summary.num_ties, "cap": cap, "ap": ap, "first": first,
                "mINP": float(summary.mINP)}
        if distmat is not None:
            info["distmat"] = distmat
        return cmc, float(summary.mAP), info

    def evaluate(self, qf: torch.Tensor, q_pids, q_camids, return_distmat: bool = False, use_cap_memo: bool = True,
                 one_call: bool = True):
        """Returns (cmc float32 ndarray [K'], mAP float, info dict).  Queries are replicated on every rank.
        `qf` may live in (pinned) host memory: it is copied on the copy stream ahead of the gallery chunks.
        On a re-ranking evaluator every query block's distances are re-ranked before they are ranked (and returned).
        one_call=False runs the staged block loop where one foreign call could do the whole evaluation (same bits)."""
        qf = _as_features(qf)
        if self.rerank:
            qf = qf.to(self.device)
            one_call = False             # the one-call path has no re-ranking stage: the staged block loop does
        if self.query_group is not None:
            with torch.cuda.device(self.device):
                self._agree_on_queries(qf)
        if qf.is_cuda:
            with torch.cuda.device(self.device):
                if qf.shape[0] > 0:
                    self._ensure_center(qf)      # one foreign call: grouping, centre, gallery pack -- the GPU is busy from here on
                elif self._gallery_dev is not None and not self.chunks:
                    self._use_center = False     # no query rows to take a centre from (and nothing to compare against)
                    self._prepare_gallery(None)
        memo_key = self._memo_key(q_pids) if use_cap_memo else None
        cap, width = _CAP_MEMO.get(memo_key, (0, 0))
        # one GPU: always one call; a sharded gallery: once the memo knows the row width the peer exchange needs
        if one_call and self._one_resident_block(qf) and (self.world == 1 or self.exchange == "peer" and width > 0):
            return self._evaluate_one_call(qf, q_pids, q_camids, return_distmat, memo_key, cap, width)
        return self._evaluate_staged(qf, q_pids, q_camids, return_distmat, memo_key, cap, width)

    def capture(self, qf: torch.Tensor, q_pids, q_camids, return_distmat: bool = False) -> "CapturedEvaluation":
        """The evaluation of one query block captured as a CUDA graph, for callers who evaluate the same shapes over and
        over: a replay costs one graph launch and one wait, with no evaluator bookkeeping, allocation or foreign call.
        Runs one ordinary evaluate() first (it fixes the centre, packs the gallery and sizes the lists), then captures
        the one-call step on a side stream with a private memory pool.  See CapturedEvaluation.

        Plain evaluation of a device-resident gallery only; ValueError for re-ranking, from_host, query_group, more
        queries than one block holds, a sharded gallery whose exchange is not "peer", and the library's debug timeline
        (ieee_set_debug_flags bit 7)."""
        qf = _as_features(qf)
        reason = self._capture_unsupported(qf.shape[0])
        if reason is not None:
            raise ValueError("capture: " + reason)
        return CapturedEvaluation(self, qf, q_pids, q_camids, return_distmat)

    def _capture_unsupported(self, Q: int) -> str | None:
        if self.query_group is not None:
            return "query_group shares GNN re-ranking across ranks; its exchanges are collectives a graph does not hold"
        if self.rerank:
            return "re-ranking ({}) runs the staged block loop, which is not captured".format(
                'rerank="gnn"' if self.gnn else "rerank=True")
        if self._gallery_dev is None:
            return "the gallery is streamed from the host (from_host); a captured step needs it in HBM"
        if self.world > 1 and self.exchange != "peer":
            return 'a sharded gallery is captured with exchange="peer" only, not {!r}'.format(self.exchange)
        if Q == 0 or self._block_rows(Q) < Q:
            return "{} queries do not make one query block ({} rows fit block_bytes={})".format(
                Q, self._block_rows_for(1 << 40, self.G), self.block_bytes)
        lib = _lib.load()
        flags = lib.ieee_set_debug_flags(0)
        lib.ieee_set_debug_flags(flags)
        if flags & 128:
            return "the library's debug timeline (ieee_set_debug_flags bit 7) records events a graph cannot hold"
        return None


class CapturedEvaluation:
    """One query block's evaluation captured as a CUDA graph (RetrievalEvaluator.capture).

    ``qf``, ``q_pids`` and ``q_camids`` are the graph's static inputs on the evaluator's device (the features in the
    dtype evaluate() computes from, the labels as int64), initialised from capture()'s arguments: copy the next query
    set into them (same shapes), then ``replay()``.  It returns what ``evaluate()`` of the evaluator returns for their
    current contents, bit for bit: (cmc, mAP, info) with ``ap``, ``first``, ``mINP``, ``num_valid``, ``num_ties``,
    ``cap`` and, when captured with ``return_distmat=True``, ``distmat``.  The tensors in ``info`` are the graph's own
    outputs: the next replay overwrites them.  ``launch()`` only enqueues the graph on the current stream and
    ``result()`` waits for that launch and parses it.

    The handle owns everything its step writes (workspace, distance block, per-query arrays, result block and its pinned
    host copy) and, on a sharded gallery, an exchange buffer of its own whose epoch lives in a device word the step
    advances itself: eager evaluations keep their own buffers and epochs.  Every rank must replay as often as the
    others, as every rank calls evaluate() alike.  When a replay's lists outgrow the captured capacity (or, sharded, the
    merged lists the row width), the result block says so; the handle then evaluates once eagerly to size the lists
    exactly, captures again and replays.  A sharded handle's exchange buffer stays allocated, as the pooled ones do."""

    def __init__(self, ev: RetrievalEvaluator, qf: torch.Tensor, q_pids, q_camids, return_distmat: bool):
        self._ev, self._return_distmat = ev, return_distmat
        dev = ev.device
        _, _, info = ev.evaluate(qf, q_pids, q_camids)
        with torch.cuda.device(dev):
            self.qf = torch.empty(qf.shape, dtype=qf.dtype, device=dev).copy_(qf)
            self.q_pids = _as_device(q_pids, torch.int64, dev).clone()
            self.q_camids = _as_device(q_camids, torch.int64, dev).clone()
            self._done = torch.cuda.Event()
        self._capture(info["cap"], ev._memo_key(q_pids))

    def _capture(self, cap: int, memo_key):
        ev, lib, dev = self._ev, _lib.load(), self._ev.device
        Q, D = self.qf.shape
        prec = _lib.PRECISIONS[ev.precision]
        k_eff = min(ev.max_rank, ev.g_total)
        with torch.cuda.device(dev):
            ex = self.epoch = None
            W = 0                                 # (no merged lists on one GPU)
            if ev.world > 1:
                # the merged lists' width the memo learnt with these labels, else the widest they can be; the ranks agree
                # on both sizes (they fix the exchange buffer's layout)
                width = _CAP_MEMO.get(memo_key, (0, 0))[1] if memo_key is not None else 0
                sizes = torch.tensor([cap, min(width, ev.world * cap) if width > 0 else ev.world * cap], device=dev)
                torch.distributed.all_reduce(sizes, op=torch.distributed.ReduceOp.MAX, group=ev.group)
                cap, W = (int(v) for v in sizes.tolist())
                self._link = PeerLink(ev.group, dev, lib.ieee_peer_exchange_bytes(Q, Q, cap, W, ev.world))
                ex = self._link.descriptor(Q, Q, Q, 0, cap, W, 0)
                self.epoch = torch.ones(1, dtype=torch.int64, device=dev)
                ws_bytes = lib.ieee_retrieve_prepared_peer_workspace_bytes(Q, D, prec, cap)
            else:
                ws_bytes = lib.ieee_retrieve_prepared_workspace_bytes(Q, D, prec, cap)
            self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            # zeroed once: the one-GPU step never writes the statistics words
            self._res = torch.zeros(96 + 4 * k_eff, dtype=torch.uint8, device=dev)
            self._host = torch.empty(self._res.numel(), dtype=torch.uint8, pin_memory=True)
            self._block = ev._new_block(Q)
            self.ap = torch.empty(Q, dtype=torch.float64, device=dev)
            self.first = torch.empty(Q, dtype=torch.int32, device=dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):         # a side stream and a private memory pool
                # the step packs the queries itself: nothing was packed ahead for the static input
                ev._one_call_launch(self.qf, self.q_pids, self.q_camids, cap, self._block, self._ws, self._res, self.ap,
                                    self.first, None, ex, self.epoch)
                self._host.copy_(self._res, non_blocking=True)
        self._graph, self._ex, self.cap, self.W = graph, ex, cap, W

    def launch(self):
        """Enqueue one replay on the current stream and return at once."""
        self._graph.replay()                     # (on the current stream of the device it was captured on)
        self._done.record(torch.cuda.current_stream(self._ev.device))

    def result(self):
        """Wait for the last launch() and return its (cmc, mAP, info)."""
        return self._finish(retry=True)

    def replay(self):
        """launch() + result()."""
        self.launch()
        return self._finish(retry=True)

    def _finish(self, retry: bool):
        self._done.synchronize()
        (overflow, longest), summary, cmc = _parse_result(self._host.numpy())
        if overflow or longest > self.W:
            if not retry:
                raise RuntimeError("ieee_b200: per-query lists overflowed an exactly sized buffer (cap=%d, longest=%d)"
                                   % (self.cap, longest))
            # exact sizes from one eager evaluation of the same contents (collective on a sharded gallery: every rank
            # sees the same statistics, so all of them get here), then a graph with those sizes
            ev = self._ev
            _, _, info = ev.evaluate(self.qf, self.q_pids, self.q_camids)
            self._capture(info["cap"], ev._memo_key(self.q_pids))
            self.launch()
            return self._finish(retry=False)
        return self._ev._result(summary, cmc, self.cap, self.ap, self.first,
                                self._block if self._return_distmat else None)


def result_lines(cmc, mAP, ranks=(1, 5, 10, 20)):
    """The result block ``Engine._evaluate`` prints (engine.py:420-425), line by line -- the format
    tools/parse_test_res.py:70-74 parses ('mAP: 61.05%', 'Rank-1  : 89.33%', ...)."""
    lines = ["** Results **", "mAP: {:.2%}".format(mAP), "CMC curve"]
    lines += ["Rank-{:<3}: {:.2%}".format(r, cmc[r - 1]) for r in ranks if r - 1 < len(cmc)]
    return lines + ["\n"]


def evaluate(qf, gf, q_pids, g_pids, q_camids, g_camids, dist_metric="euclidean", normalize_feature=False, rerank=False,
             ranks=(1, 5, 10, 20), max_rank=20, precision=None, verbose=True, dataset_name=""):
    """Tail of ``Engine._evaluate`` (engine.py:391-441) on one GPU.  Feature tensors may live on the host
    (copied once) or on the device.  Prints the reference's result lines (engine.py:420-425), which
    tools/parse_test_res.py:70 parses, and returns (cmc, mAP)."""
    _lib.require_cuda()
    dev = qf.device if qf.is_cuda else torch.device("cuda", torch.cuda.current_device())
    streamed = (not rerank) and (not gf.is_cuda)
    if not streamed:
        qf = qf.to(dev, non_blocking=True)
        gf = gf.to(dev, non_blocking=True)
    if verbose and normalize_feature:
        print("Normalzing features with L2 norm ...")
    if verbose:
        print("Computing distance matrix with metric={} ...".format(dist_metric))
    if streamed:
        ev = RetrievalEvaluator.from_host(gf, g_pids, g_camids, dist_metric, normalize_feature, precision, max_rank)
        cmc, mAP, _ = ev.evaluate(qf, q_pids, q_camids)
    elif not rerank:
        ev = RetrievalEvaluator(gf, g_pids, g_camids, dist_metric, normalize_feature, precision, max_rank)
        cmc, mAP, _ = ev.evaluate(qf, q_pids, q_camids)
    elif rerank == "gnn":
        # alternative re-ranking mode (torchreid/utils/GPU-Re-Ranking/gnn_reranking.py:27-59; its driver L2-normalises
        # the features and uses k1 = 26, k2 = 7): the negated re-ranked similarity ranks like a distance matrix
        from .metrics.rank import evaluate_device
        from .utils.gnn_reranking import gnn_reranking_distmat
        if verbose:
            print("Applying GNN re-ranking ...")
        norm = torch.nn.functional.normalize
        distmat = gnn_reranking_distmat(norm(qf.float(), dim=1), norm(gf.float(), dim=1), 26, 7)
        cmc_t, summary, _ = evaluate_device(distmat, q_pids, g_pids, q_camids, g_camids, max_rank)
        raise_for_status(summary, max_rank)
        cmc, mAP = cmc_t.cpu().numpy(), float(summary.mAP)
    else:
        from .metrics.distance import _device_distmat
        from .metrics.rank import evaluate_device
        if verbose:
            print("Applying person re-ranking ...")
        qg = _device_distmat(qf, gf, dist_metric, normalize_feature, precision)
        qq = _device_distmat(qf, qf, dist_metric, normalize_feature, precision)
        gg = _device_distmat(gf, gf, dist_metric, normalize_feature, precision)
        distmat = re_ranking_device(qg, qq, gg)
        cmc_t, summary, _ = evaluate_device(distmat, q_pids, g_pids, q_camids, g_camids, max_rank)
        raise_for_status(summary, max_rank)
        cmc, mAP = cmc_t.cpu().numpy(), float(summary.mAP)
    if verbose:
        print("Computing CMC and mAP for {}".format(dataset_name))
        for line in result_lines(cmc, mAP, ranks):
            print(line)
    return cmc, mAP
