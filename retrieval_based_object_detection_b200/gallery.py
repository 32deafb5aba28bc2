"""Device-resident gallery: the Python face of one ``rbod_gallery`` handle (include/rbod.h).

A ``Gallery`` is what a collection's vectors live in.  Host data comes in as numpy arrays, device
data as torch CUDA tensors (only their ``data_ptr()`` crosses the C ABI); results come back in the
kind the queries were given in.  Every method is a thin call into librbod.so -- there is no Python
or CPU implementation of the arithmetic here.

Reference call sites served (paths in the reference repo): upsert <- 31_…py:178-179, 32_…py:41-42;
get_rows <- scroll(with_vectors=True) 32_…py:123-137, 33_…py:96-110; segment_mean <-
compute_average 32_…py:9-10; search <- cosine_similarity 33_…py:76-77,151 (Q x N top-k).
"""
from __future__ import annotations

import ctypes
import sys
from dataclasses import dataclass

import numpy as np

from . import _native as N


@dataclass
class SearchResult:
    scores: object      # [Q, k] float32: cosine / dot descending, or distance ascending (euclid, manhattan)
    rows: object        # [Q, k] int64 row slots, -1 = no result
    scores64: object    # [Q, k] float64 (None unless requested)
    stats: dict


def _is_torch(x) -> bool:
    return "torch" in sys.modules and isinstance(x, sys.modules["torch"].Tensor)


def _current_stream() -> int:
    torch = sys.modules.get("torch")
    if torch is not None and torch.cuda.is_available() and torch.cuda.is_initialized():
        return int(torch.cuda.current_stream().cuda_stream)
    return 0


def _as_host(x, dtype) -> np.ndarray:
    return np.ascontiguousarray(x, dtype=dtype)


class Gallery:
    """One collection's vectors on one GPU."""

    def __init__(self, dim: int, dtype: str = "f32", metric: str = "cosine", capacity: int = 0, device: int = 0):
        self._lib = N.load()
        self._h = ctypes.c_void_p()
        self.dim = int(dim)
        self.dtype = dtype
        self.metric = metric
        self.device = int(device)
        self.options = {}     # what set_option was given
        N.check(self._lib.rbod_create(self.dim, N.DTYPES[dtype], N.METRICS[metric], int(capacity), self.device,
                                      ctypes.byref(self._h)))

    # -- lifetime ---------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.rbod_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self) -> int:
        return int(self._lib.rbod_count(self._h))

    @property
    def count(self) -> int:
        return len(self)

    def info(self) -> dict:
        gi = N.GalleryInfo()
        N.check(self._lib.rbod_info(self._h, ctypes.byref(gi)))
        return {f: getattr(gi, f) for f, _ in gi._fields_}

    def truncate(self, rows: int) -> None:
        N.check(self._lib.rbod_truncate(self._h, int(rows)))

    def set_option(self, key: str, value: int) -> None:
        N.check(self._lib.rbod_set_option(self._h, key.encode(), int(value)))
        self.options[key] = int(value)

    # -- pointer plumbing -------------------------------------------------------------------
    def _in(self, x, dtype_np, dtype_name: str):
        """-> (object to keep alive, raw pointer)."""
        if x is None:
            return None, None
        if _is_torch(x):
            torch = sys.modules["torch"]
            want = getattr(torch, dtype_name)
            if x.dtype != want or not x.is_contiguous():
                x = x.to(want).contiguous()
            return x, x.data_ptr()
        a = _as_host(x, dtype_np)
        return a, a.ctypes.data

    def _alloc_like(self, like, shape, dtype_np, dtype_name: str):
        if _is_torch(like) and like.is_cuda:
            torch = sys.modules["torch"]
            t = torch.empty(shape, dtype=getattr(torch, dtype_name), device=like.device)
            return t, t.data_ptr()
        a = np.empty(shape, dtype=dtype_np)
        return a, a.ctypes.data

    # -- K1 ---------------------------------------------------------------------------------
    def upsert(self, rows, slots=None, return_norms: bool = False, raw: bool = False, stream=None):
        """Normalise (COSINE) and store ``rows`` [n, dim] at ``slots`` (None = append)."""
        keep, p_rows = self._in(rows, np.float32, "float32")
        shape = tuple(keep.shape)
        if len(shape) == 1:
            shape = (1, shape[0])
        if len(shape) != 2 or shape[1] != self.dim:
            raise ValueError(f"upsert: expected [n, {self.dim}] rows, got {tuple(keep.shape)}")
        n = shape[0]
        slots_a = None if slots is None else _as_host(slots, np.int64)
        if slots_a is not None and slots_a.shape != (n,):
            raise ValueError("upsert: slots must have one entry per row")
        norms, p_norms = (self._alloc_like(keep, (n,), np.float32, "float32") if return_norms else (None, None))
        N.check(self._lib.rbod_upsert(self._h, p_rows, n, None if slots_a is None else slots_a.ctypes.data, p_norms,
                                      N.RBOD_UPSERT_RAW if raw else 0, stream if stream is not None else _current_stream()))
        return norms

    def get_rows(self, rows):
        """Stored rows widened to float32."""
        keep, p_idx = self._in(rows, np.int64, "int64")
        n = int(keep.shape[0])
        out, p_out = self._alloc_like(keep, (n, self.dim), np.float32, "float32")
        N.check(self._lib.rbod_get_rows(self._h, p_idx, n, p_out, _current_stream()))
        return out

    # -- K2 ---------------------------------------------------------------------------------
    def segment_mean(self, offsets, row_idx=None):
        """Per-class normalised mean ("average" delegate) of stored rows; CSR ``offsets`` [C+1]."""
        k_off, p_off = self._in(offsets, np.int64, "int64")
        k_idx, p_idx = self._in(row_idx, np.int64, "int64")
        C = int(k_off.shape[0]) - 1
        if C < 0:
            raise ValueError("segment_mean: offsets must have at least one entry")
        out, p_out = self._alloc_like(k_off, (C, self.dim), np.float32, "float32")
        N.check(self._lib.rbod_segment_mean(self._h, p_idx, p_off, C, p_out, _current_stream()))
        return out

    def segment_sums(self, offsets, row_idx=None):
        """Raw per-class float64 column sums [C, dim] of this shard's stored rows as a torch CUDA tensor -- the
        local half of the sharded delegate build (``ShardedGallery.segment_mean`` all-reduces and finishes them)."""
        torch = sys.modules.get("torch")
        if torch is None:
            import torch
        k_off, p_off = self._in(offsets, np.int64, "int64")
        k_idx, p_idx = self._in(row_idx, np.int64, "int64")
        C = int(k_off.shape[0]) - 1
        if C < 0:
            raise ValueError("segment_sums: offsets must have at least one entry")
        out = torch.empty((C, self.dim), dtype=torch.float64, device=torch.device("cuda", self.device))
        N.check(self._lib.rbod_segment_sums(self._h, p_idx, p_off, C, out.data_ptr(), _current_stream()))
        return out

    def segment_delegates(self, kind: str, offsets, row_idx=None, alpha: float = 2.0):
        """Per-class delegate of ``kind`` in {"average", "centroid", "weighted", "medoid"}
        (32_create_delegate_vector.py:9-26) in stored form -> (vectors [C, dim] float32, member rows [C] int64,
        -1 where the delegate is not a member)."""
        if kind not in N.DELEGATE_KINDS:
            raise ValueError(f"unknown delegate kind {kind!r}")
        k_off, p_off = self._in(offsets, np.int64, "int64")
        k_idx, p_idx = self._in(row_idx, np.int64, "int64")
        C = int(k_off.shape[0]) - 1
        if C < 0:
            raise ValueError("segment_delegates: offsets must have at least one entry")
        out, p_out = self._alloc_like(k_off, (C, self.dim), np.float32, "float32")
        mem, p_mem = self._alloc_like(k_off, (C,), np.int64, "int64")
        N.check(self._lib.rbod_segment_delegates(self._h, N.DELEGATE_KINDS[kind], p_idx, p_off, C, float(alpha), p_out,
                                                 p_mem, _current_stream()))
        return out, mem

    # -- K3 ---------------------------------------------------------------------------------
    def search(self, queries, k: int, row_mask=None, want_scores64: bool = False, out=None, stream=None,
               mask_of_query=None) -> SearchResult:
        """Exact top-k of ``queries`` [Q, dim] against the stored rows under the collection's distance (cosine by
        default; ``scores64`` carries the ordering key -d^2 / -d for euclid / manhattan collections).

        ``row_mask``: uint32 row bitmask (bit r % 32 of word r // 32 = row r allowed) shared by every query.  With
        ``mask_of_query`` [Q] int32 (the mask each query uses, -1 = no filter), ``row_mask`` is [M, words] instead:
        one mask per distinct filter, all answered in one pass (rbod_search_masks)."""
        keep, p_q = self._in(queries, np.float32, "float32")
        if keep.ndim == 1:
            keep = keep.reshape(1, -1)
        if keep.ndim != 2 or keep.shape[1] != self.dim:
            raise ValueError(f"search: expected [Q, {self.dim}] queries, got {tuple(keep.shape)}")
        Q = int(keep.shape[0])
        k_mask, p_mask = self._in(row_mask, np.uint32, "int32")
        k_ids, p_ids = self._in(mask_of_query, np.int32, "int32")
        n_masks = 0
        if k_ids is not None:
            if tuple(k_ids.shape) != (Q,):
                raise ValueError(f"search: mask_of_query must hold one mask id per query ({Q}), got {tuple(k_ids.shape)}")
            if k_mask is not None:
                words = (len(self) + 31) // 32
                if k_mask.ndim != 2 or k_mask.shape[1] != words:
                    raise ValueError(f"search: with mask_of_query, row_mask must be [M, {words}] words, "
                                     f"got {tuple(k_mask.shape)}")
                n_masks = int(k_mask.shape[0])
        if out is not None:
            scores, rows = out[0], out[1]
            s64 = out[2] if len(out) > 2 else None
            p_s = scores.data_ptr() if _is_torch(scores) else scores.ctypes.data
            p_r = rows.data_ptr() if _is_torch(rows) else rows.ctypes.data
            p_64 = None if s64 is None else (s64.data_ptr() if _is_torch(s64) else s64.ctypes.data)
        else:
            scores, p_s = self._alloc_like(keep, (Q, k), np.float32, "float32")
            rows, p_r = self._alloc_like(keep, (Q, k), np.int64, "int64")
            s64, p_64 = (self._alloc_like(keep, (Q, k), np.float64, "float64") if want_scores64 else (None, None))
        st = N.SearchStats()
        stream = stream if stream is not None else _current_stream()
        if k_ids is not None:
            N.check(self._lib.rbod_search_masks(self._h, p_q, Q, int(k), p_mask, n_masks, p_ids, p_s, p_r, p_64,
                                                ctypes.byref(st), stream))
        else:
            N.check(self._lib.rbod_search(self._h, p_q, Q, int(k), p_mask, p_s, p_r, p_64, ctypes.byref(st), stream))
        stats = {f: getattr(st, f) for f, _ in st._fields_}
        return SearchResult(scores, rows, s64, stats)

    # -- K8 ---------------------------------------------------------------------------------
    def search_mmr(self, queries, limit: int, candidates: int, diversity, score_threshold=None, row_mask=None,
                   mask_of_query=None, want_keys: bool = False) -> SearchResult:
        """Maximal marginal relevance (rbod_search_mmr): per query, the exact top-``candidates`` c_0 .. c_{L-1} of an
        ordinary search, then ``limit`` of them picked greedily.  With the collection's fp64 search key, sim = identity
        (-sqrt(-key) for euclid), rel(c) = sim(key(query, c)) and lambda = 1 - diversity, the first pick is c_0 and every
        later pick maximises lambda * rel(c) - diversity * max over picked s of sim(key(s, c)) (fp64, in that order),
        exact ties to the smaller candidate rank.  Qdrant >= 1.15 documents the same kind of rule; this one has not been
        checked against a live Qdrant or its source.

        ``diversity``: a float in [0, 1] or one per query.  ``score_threshold``: None, a float or one per query (NaN =
        none): only candidates whose search score is >= it (<= for euclid / manhattan distances) take part.
        ``row_mask`` / ``mask_of_query``: as ``search``.  -> ``scores`` [Q, limit] float32 search scores and ``rows``
        [Q, limit] int64 in SELECTION order (padded with -inf / +inf for distances, and -1), ``scores64`` the fp64 keys
        when ``want_keys``."""
        keep, p_q = self._in(queries, np.float32, "float32")
        if keep.ndim == 1:
            keep = keep.reshape(1, -1)
        if keep.ndim != 2 or keep.shape[1] != self.dim:
            raise ValueError(f"search_mmr: expected [Q, {self.dim}] queries, got {tuple(keep.shape)}")
        Q = int(keep.shape[0])
        div = np.ascontiguousarray(np.broadcast_to(np.asarray(diversity, dtype=np.float64), (Q,)))
        thr = (None if score_threshold is None else
               np.ascontiguousarray(np.broadcast_to(np.asarray(score_threshold, dtype=np.float32), (Q,))))
        k_mask, p_mask = self._in(row_mask, np.uint32, "int32")
        k_ids, p_ids = self._in(mask_of_query, np.int32, "int32")
        n_masks = 0 if k_mask is None else 1
        if k_ids is not None:
            if tuple(k_ids.shape) != (Q,):
                raise ValueError(f"search_mmr: mask_of_query must hold one mask id per query ({Q})")
            n_masks = 0
            if k_mask is not None:
                words = (len(self) + 31) // 32
                if k_mask.ndim != 2 or k_mask.shape[1] != words:
                    raise ValueError(f"search_mmr: with mask_of_query, row_mask must be [M, {words}] words, "
                                     f"got {tuple(k_mask.shape)}")
                n_masks = int(k_mask.shape[0])
        scores, p_s = self._alloc_like(keep, (Q, limit), np.float32, "float32")
        rows, p_r = self._alloc_like(keep, (Q, limit), np.int64, "int64")
        keys, p_k = (self._alloc_like(keep, (Q, limit), np.float64, "float64") if want_keys else (None, None))
        st = N.SearchStats()
        N.check(self._lib.rbod_search_mmr(self._h, p_q, Q, int(limit), int(candidates), div.ctypes.data,
                                          None if thr is None else thr.ctypes.data, p_mask, n_masks, p_ids, p_s, p_r,
                                          p_k, ctypes.byref(st), _current_stream()))
        return SearchResult(scores, rows, keys, {f: getattr(st, f) for f, _ in st._fields_})

    # -- K6 ---------------------------------------------------------------------------------
    def recommend(self, examples, signs, offsets, k: int, row_mask=None, mask_of_request=None,
                  want_keys: bool = False) -> SearchResult:
        """Exact best_score recommendation (rbod_recommend): request r is the examples ``offsets[r]:offsets[r + 1]`` of
        ``examples`` [E, dim], each positive (``signs`` +1) or negative (-1), 1 to 32 per request.  A row's score is
        s(sim(bp)) when its best positive key bp beats its best negative key bn, else -s(sim(bn)), with the search key
        of the collection's metric, sim = identity (-sqrt(-key) for euclid) and s(y) = 0.5 (y / (1 + |y|) + 1): the
        best_score rule of Qdrant >= 1.7, not checked against a live Qdrant.  Larger is better for every metric.

        -> ``scores`` [R, k] float32 descending (-inf padded), ``rows`` [R, k] int64 (-1 padded), ``scores64`` the fp64
        scores when ``want_keys``.  ``row_mask`` / ``mask_of_request`` are as ``search``'s ``row_mask`` /
        ``mask_of_query``, one mask id per request."""
        return self._example_search("recommend", "signs", examples, signs, offsets, k, row_mask, mask_of_request,
                                    want_keys)

    # -- K7 ---------------------------------------------------------------------------------
    def discover(self, examples, roles, offsets, k: int, row_mask=None, mask_of_request=None,
                 want_keys: bool = False) -> SearchResult:
        """Exact discovery and context search (rbod_discover): request r is the examples ``offsets[r]:offsets[r + 1]``
        of ``examples`` [E, dim], 1 to 32 per request: an optional target first (``roles`` 0), then pairs of a positive
        (+1) directly followed by its negative (-1).  With the search key of the collection's metric, sim = identity
        (-sqrt(-key) for euclid), f(y) = y / (1 + |y|), s(y) = 0.5 (f(y) + 1) and MARGIN = 2**-23, a row scores

        * with a target t (discovery): sum over pairs of (+1 if key(p) > key(n) else -1) + s(sim(key(t)));
        * without (context): sum over pairs, in order, of f(min(sim(key(p)) - sim(key(n)) - MARGIN, 0)), which is 0
          for every row on the positive side of every pair.

        This is the rule of Qdrant >= 1.7 as read from its source, not checked against a live Qdrant.  Larger is better
        for every metric.  Returns and masks as ``recommend``."""
        return self._example_search("discover", "roles", examples, roles, offsets, k, row_mask, mask_of_request,
                                    want_keys)

    def _example_search(self, name, what, examples, per_example, offsets, k, row_mask, mask_of_request, want_keys):
        """rbod_recommend / rbod_discover (``name``) with ``per_example`` the int8 signs / roles (``what``)."""
        keep, p_x = self._in(examples, np.float32, "float32")
        if keep.ndim != 2 or keep.shape[1] != self.dim:
            raise ValueError(f"{name}: expected [E, {self.dim}] examples, got {tuple(keep.shape)}")
        sg = _as_host(per_example, np.int8)
        off = _as_host(offsets, np.int64)
        if off.ndim != 1 or len(off) < 1 or sg.shape != (int(keep.shape[0]),):
            raise ValueError(f"{name}: offsets must be [R + 1] and {what} [E]")
        R = len(off) - 1
        k_mask, p_mask = self._in(row_mask, np.uint32, "int32")
        k_ids, p_ids = self._in(mask_of_request, np.int32, "int32")
        n_masks = 0 if k_mask is None else 1
        if k_ids is not None:
            if tuple(k_ids.shape) != (R,):
                raise ValueError(f"{name}: mask_of_request must hold one mask id per request ({R})")
            n_masks = 0
            if k_mask is not None:
                words = (len(self) + 31) // 32
                if k_mask.ndim != 2 or k_mask.shape[1] != words:
                    raise ValueError(f"{name}: with mask_of_request, row_mask must be [M, {words}] words, "
                                     f"got {tuple(k_mask.shape)}")
                n_masks = int(k_mask.shape[0])
        scores, p_s = self._alloc_like(keep, (R, k), np.float32, "float32")
        rows, p_r = self._alloc_like(keep, (R, k), np.int64, "int64")
        keys, p_k = (self._alloc_like(keep, (R, k), np.float64, "float64") if want_keys else (None, None))
        st = N.SearchStats()
        N.check(getattr(self._lib, "rbod_" + name)(self._h, p_x, int(keep.shape[0]), sg.ctypes.data, off.ctypes.data, R,
                                                 int(k), p_mask, n_masks, p_ids, p_s, p_r, p_k, ctypes.byref(st),
                                                 _current_stream()))
        return SearchResult(scores, rows, keys, {f: getattr(st, f) for f, _ in st._fields_})

    # -- split search (row-sharded collections): see include/rbod.h "Split search" ------------------------------
    def search_begin(self, queries, k: int, approx_m: int, out_approx, row_mask=None, stream=None) -> dict:
        """First half: K3 + selection; fills ``out_approx`` [Q, approx_m + 1] float32 (torch CUDA tensor) with this
        shard's best approximate scores and its error bound.  Device ``queries`` must stay alive until search_end."""
        keep, p_q = self._in(queries, np.float32, "float32")
        if keep.ndim != 2 or keep.shape[1] != self.dim:
            raise ValueError(f"search_begin: expected [Q, {self.dim}] queries, got {tuple(keep.shape)}")
        Q = int(keep.shape[0])
        if tuple(out_approx.shape) != (Q, approx_m + 1) or not out_approx.is_contiguous():
            raise ValueError("search_begin: out_approx must be a contiguous [Q, approx_m + 1] float32 tensor")
        k_mask, p_mask = self._in(row_mask, np.uint32, "int32")
        st = N.SearchStats()
        N.check(self._lib.rbod_search_begin(self._h, p_q, Q, int(k), int(approx_m), p_mask, out_approx.data_ptr(),
                                            ctypes.byref(st), stream if stream is not None else _current_stream()))
        self._pending_queries = keep
        return {f: getattr(st, f) for f, _ in st._fields_}

    def search_end(self, cut, k: int, packed, stream=None) -> dict:
        """Second half: ``cut`` [Q, 2] float32 from global_cut; ``packed`` = ONE contiguous int64 CUDA tensor of
        2*Q*k + Q words that receives [Q,k] float64 scores, [Q,k] local row slots and the [Q] float64 bounds."""
        Q = int(cut.shape[0])
        if packed.numel() != 2 * Q * k + Q or not packed.is_contiguous():
            raise ValueError("search_end: packed must hold 2*Q*k + Q 8-byte words")
        base = packed.data_ptr()
        st = N.SearchStats()
        N.check(self._lib.rbod_search_end(self._h, cut.data_ptr(), Q, int(k), base, base + 8 * Q * k, base + 16 * Q * k,
                                          ctypes.byref(st), stream if stream is not None else _current_stream()))
        self._pending_queries = None
        return {f: getattr(st, f) for f, _ in st._fields_}

    def last_k3_ms(self) -> float:
        out = ctypes.c_float()
        N.check(self._lib.rbod_last_k3_ms(self._h, ctypes.byref(out)))
        return float(out.value)

    def debug_profile(self) -> dict:
        """Wait-cycle counters of the K3 launches since the last call (needs set_option("k3_prof", 1)); clears them."""
        out = (ctypes.c_int64 * 16)()
        N.check(self._lib.rbod_debug_profile(self._h, out))
        names = ("prod_wait_empty", "prod_wait_throttle", "mma_wait_query_tile", "mma_wait_accumulator", "mma_wait_data",
                 "epi_wait_accumulator", "epi_prune", "cta_cycles", "ctas", "epi_warps", "prunes", "prod_wait_empty_follower",
                 "prod_issue", "mma_issue")
        return dict(zip(names, list(out)))

    def debug_scores(self, queries):
        """Raw scores of the tcgen05 pass (test hook): [Q, rows] float32."""
        keep, p_q = self._in(queries, np.float32, "float32")
        Q = int(keep.shape[0])
        out, p_out = self._alloc_like(keep, (Q, len(self)), np.float32, "float32")
        N.check(self._lib.rbod_debug_scores(self._h, p_q, Q, p_out, _current_stream()))
        return out


def merge_topk(scores64, ids, k: int, stream=None):
    """K4: [G, Q, k] gathered per-shard lists (torch CUDA tensors) -> global top-k (scores, ids, scores64)."""
    torch = sys.modules["torch"]
    lib = N.load()
    G, Q, kk = scores64.shape
    if kk != k:
        raise ValueError("merge_topk: last dimension must equal k")
    scores64 = scores64.contiguous()
    ids = ids.contiguous()
    out_s = torch.empty((Q, k), dtype=torch.float32, device=scores64.device)
    out_i = torch.empty((Q, k), dtype=torch.int64, device=scores64.device)
    out_d = torch.empty((Q, k), dtype=torch.float64, device=scores64.device)
    N.check(lib.rbod_merge_topk(scores64.data_ptr(), ids.data_ptr(), G, Q, k, out_s.data_ptr(), out_i.data_ptr(),
                                out_d.data_ptr(), stream if stream is not None else _current_stream()))
    return out_s, out_i, out_d


def merge_topk_packed(gathered, shard_row0, k: int, stream=None):
    """K4 over ONE gathered buffer: ``gathered`` [G, 2, Q, k] int64 words on the device, where [:, 0] holds each
    shard's float64 scores (bit pattern) and [:, 1] its LOCAL row slots; ``shard_row0`` = the G global row offsets.
    -> (scores f32, global ids i64, scores f64), each [Q, k]."""
    torch = sys.modules["torch"]
    lib = N.load()
    G, two, Q, kk = gathered.shape
    if two != 2 or kk != k:
        raise ValueError("merge_topk_packed: expected a [G, 2, Q, k] buffer")
    gathered = gathered.contiguous()
    row0 = np.ascontiguousarray(shard_row0, dtype=np.int64)
    if row0.shape != (G,):
        raise ValueError("merge_topk_packed: one row offset per shard")
    out_s = torch.empty((Q, k), dtype=torch.float32, device=gathered.device)
    out_i = torch.empty((Q, k), dtype=torch.int64, device=gathered.device)
    out_d = torch.empty((Q, k), dtype=torch.float64, device=gathered.device)
    N.check(lib.rbod_merge_topk_packed(gathered.data_ptr(), row0.ctypes.data, G, Q, k, out_s.data_ptr(),
                                       out_i.data_ptr(), out_d.data_ptr(),
                                       stream if stream is not None else _current_stream()))
    return out_s, out_i, out_d


def global_cut(gathered_approx, k: int, stream=None):
    """[G, Q, m + 1] gathered search_begin outputs (float32, CUDA) -> [Q, 2] {global k-th best approximate score,
    largest error bound}."""
    torch = sys.modules["torch"]
    lib = N.load()
    G, Q, m1 = gathered_approx.shape
    gathered_approx = gathered_approx.contiguous()
    out = torch.empty((Q, 2), dtype=torch.float32, device=gathered_approx.device)
    N.check(lib.rbod_global_cut(gathered_approx.data_ptr(), G, Q, m1 - 1, int(k), out.data_ptr(),
                                stream if stream is not None else _current_stream()))
    return out


def merge_topk_certified(gathered, shard_row0, Q: int, k: int, stream=None):
    """K4 + certification over the gathered search_end buffers: ``gathered`` [G, 2*Q*k + Q] int64 words (CUDA).
    -> (scores f32, global ids, scores f64, flag_q int32 [Q], n_flag int32 [1]); flag_q[:n_flag] are the queries whose
    merged answer is not certified (to be answered by a full search)."""
    torch = sys.modules["torch"]
    lib = N.load()
    G, words = gathered.shape
    if words != 2 * Q * k + Q:
        raise ValueError("merge_topk_certified: expected [G, 2*Q*k + Q] words")
    gathered = gathered.contiguous()
    row0 = np.ascontiguousarray(shard_row0, dtype=np.int64)
    if row0.shape != (G,):
        raise ValueError("merge_topk_certified: one row offset per shard")
    dev = gathered.device
    out_s = torch.empty((Q, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((Q, k), dtype=torch.int64, device=dev)
    out_d = torch.empty((Q, k), dtype=torch.float64, device=dev)
    flag_q = torch.empty((Q,), dtype=torch.int32, device=dev)
    n_flag = torch.empty((1,), dtype=torch.int32, device=dev)
    N.check(lib.rbod_merge_topk_certified(gathered.data_ptr(), row0.ctypes.data, G, Q, k, out_s.data_ptr(),
                                          out_i.data_ptr(), out_d.data_ptr(), flag_q.data_ptr(), n_flag.data_ptr(),
                                          stream if stream is not None else _current_stream()))
    return out_s, out_i, out_d, flag_q, n_flag


def segment_finish(sums, counts, normalize: bool = True, stream=None):
    """sums [C, dim] float64 and counts [C] int64 (torch CUDA tensors, already reduced over the shards) ->
    delegate vectors [C, dim] float32: fp32(sum / count), L2-normalised for COSINE collections."""
    torch = sys.modules["torch"]
    lib = N.load()
    sums = sums.to(torch.float64).contiguous()
    counts = counts.to(torch.int64).contiguous()
    C, dim = sums.shape
    if counts.shape != (C,):
        raise ValueError("segment_finish: counts must have one entry per class")
    out = torch.empty((C, dim), dtype=torch.float32, device=sums.device)
    N.check(lib.rbod_segment_finish(sums.data_ptr(), counts.data_ptr(), C, dim, 1 if normalize else 0, out.data_ptr(),
                                    stream if stream is not None else _current_stream()))
    return out


def l2norm_pack(x, out_dtype: str = "bf16", want_norms: bool = False):
    """K1 on caller-owned CUDA tensors: x [n, dim] float32 -> normalised rows of ``out_dtype``."""
    torch = sys.modules["torch"]
    lib = N.load()
    x = x.contiguous()
    n, dim = x.shape
    tdt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[out_dtype]
    out = torch.empty((n, dim), dtype=tdt, device=x.device)
    norms = torch.empty((n,), dtype=torch.float32, device=x.device) if want_norms else None
    N.check(lib.rbod_l2norm_pack(x.data_ptr(), n, dim, N.DTYPES[out_dtype], out.data_ptr(), dim,
                                 None if norms is None else norms.data_ptr(), _current_stream()))
    return (out, norms) if want_norms else out
