"""Drop-in ``qdrant_client`` for dmweapon/Retrieval_based_object_detection, backed by librbod.so.

The reference scripts do ``from qdrant_client import QdrantClient`` and talk to a Qdrant server
(util/qdrant_manager.py:1, 31_…py:19, 32_…py:5, 33_…py:12).  With this package first on
``sys.path`` the same scripts run unchanged: the "server" becomes a directory on disk
(``$RBOD_STORE_DIR/<host>_<port>``, default ``~/.rbod/store``) plus a B200-resident gallery, and
every vector operation (normalise-on-upsert, stored-vector reads, delegate means, cosine top-k)
is a call through the C ABI in include/rbod.h.  There is no CPU implementation of those
operations: without the built extension and a B200 they raise.

Method subset = what the four scripts call (SURVEY.md §8(b)) + ``search`` / ``query_points`` /
``search_batch`` as BASELINE.json's north star specifies, + ``recommend`` / ``recommend_batch``, + ``discover`` /
``discover_batch`` and ``query_points(query=DiscoverQuery | ContextQuery)``, + ``query_points(query=NearestQuery(mmr=...))``
and ``query_batch_points``.  Configuration is by environment only,
because the scripts take no flags: ``RBOD_STORE_DIR``, ``RBOD_GALLERY_DTYPE`` (f32 | bf16 | f16),
``RBOD_DEVICE`` (CUDA ordinal).
"""
from __future__ import annotations

import atexit
import os
import uuid
from typing import Any, Dict, Iterable, List, Optional, Sequence

import numpy as np

from retrieval_based_object_detection_b200.store import Collection, CollectionNotFound, StoreRoot, canonical_id

from . import models
from .models import (Batch, CollectionConfig, CollectionDescription, CollectionInfo, CollectionParams,
                     CollectionsResponse, ContextExamplePair, ContextPair, ContextQuery, CountResult,
                     DiscoverQuery, DiscoverRequest, Distance, NearestQuery, PointStruct, QueryRequest, QueryResponse,
                     RecommendQuery, RecommendRequest, RecommendStrategy, Record, ScoredPoint, SearchRequest,
                     UpdateResult, UpdateStatus, VectorParams)

__all__ = ["QdrantClient", "models", "CollectionNotFound"]
__version__ = "1.9.0+rbod"

_ROOTS: Dict[str, StoreRoot] = {}


def _close_all() -> None:
    for root in list(_ROOTS.values()):
        try:
            root.close()
        except Exception:  # pragma: no cover - interpreter shutdown
            pass
    _ROOTS.clear()


atexit.register(_close_all)


def _distance_name(d) -> str:
    if isinstance(d, Distance):
        return d.value
    for cand in Distance:
        if str(d).lower() in (cand.value.lower(), cand.name.lower()):
            return cand.value
    raise ValueError(f"unknown distance {d!r}")


MAX_MMR_CANDIDATES = 1024   # candidates_limit of an MMR query (rbod_search_mmr)


def _context_pairs(context) -> list:
    """A discovery ``context`` -> [(positive, negative)].  ``context`` is None, one pair or a list of pairs; a pair is a
    ``ContextExamplePair``, a ``ContextPair`` or a (positive, negative) tuple (a 2-tuple whose members are neither
    pair models nor 2-tuples)."""
    models_ = (ContextExamplePair, ContextPair)

    def is_pair(p):
        return isinstance(p, models_) or (isinstance(p, tuple) and len(p) == 2 and not any(
            isinstance(x, models_) or (isinstance(x, tuple) and len(x) == 2) for x in p))

    if context is None:
        return []
    out = []
    for p in ([context] if is_pair(context) else list(context)):
        if not is_pair(p):
            raise ValueError(f"discover: a context pair is a ContextExamplePair, a ContextPair or a (positive, negative) "
                             f"tuple, got {p!r}")
        out.append((p.positive, p.negative) if isinstance(p, models_) else p)
    return out


class QdrantClient:
    """The client class the reference scripts instantiate as ``QdrantClient(host=..., port=...)``."""

    def __init__(self, location: Optional[str] = None, url: Optional[str] = None, port: Optional[int] = 6333,
                 host: Optional[str] = None, path: Optional[str] = None, **_ignored: Any):
        dtype = os.environ.get("RBOD_GALLERY_DTYPE", "f32")
        device = int(os.environ.get("RBOD_DEVICE", "0"))
        if location == ":memory:":
            self._root = StoreRoot(None, dtype, device)
            self._key = None
            return
        if path is not None:
            directory = os.path.abspath(path)
        else:
            if url is not None:
                hostport = url.split("://", 1)[-1].rstrip("/")
                host, _, p = hostport.partition(":")
                port = int(p) if p else port
            host = host or location or "localhost"
            if not isinstance(port, int):
                raise ValueError(f"port must be an int, got {port!r}")
            base = os.environ.get("RBOD_STORE_DIR") or os.path.join(os.path.expanduser("~"), ".rbod", "store")
            directory = os.path.join(os.path.abspath(base), f"{host}_{port}")
        self._key = directory
        root = _ROOTS.get(directory)
        if root is None:
            root = StoreRoot(directory, dtype, device)
            _ROOTS[directory] = root
        self._root = root

    # ------------------------------------------------------------------ collections
    def get_collections(self) -> CollectionsResponse:
        return CollectionsResponse(collections=[CollectionDescription(name=n) for n in self._root.names()])

    def collection_exists(self, collection_name: str) -> bool:
        return self._root.exists(collection_name)

    def get_collection(self, collection_name: str) -> CollectionInfo:
        col = self._root.get(collection_name)
        params = CollectionParams(vectors=VectorParams(size=col.dim, distance=Distance(col.distance)))
        return CollectionInfo(points_count=len(col), vectors_count=len(col), indexed_vectors_count=len(col),
                              config=CollectionConfig(params=params))

    def _vector_params(self, vectors_config) -> VectorParams:
        if isinstance(vectors_config, dict):
            if set(vectors_config) == {"size", "distance"}:
                return VectorParams(**vectors_config)
            raise ValueError("named vectors are not supported by this drop-in")
        if not hasattr(vectors_config, "size") or not hasattr(vectors_config, "distance"):
            raise ValueError("vectors_config must be VectorParams(size=..., distance=...)")
        return vectors_config

    def create_collection(self, collection_name: str, vectors_config=None, **_ignored: Any) -> bool:
        vp = self._vector_params(vectors_config)
        size = int(vp.size)
        if size < 1 or size > 65536:
            raise ValueError(f"vector size {size} out of range")
        self._root.create(collection_name, size, _distance_name(vp.distance))
        return True

    def recreate_collection(self, collection_name: str, vectors_config=None, **kwargs: Any) -> bool:
        # util/qdrant_manager.py:82-85 -- drop if present, then create empty
        self._vector_params(vectors_config)
        self._root.delete(collection_name)
        return self.create_collection(collection_name, vectors_config, **kwargs)

    def delete_collection(self, collection_name: str, **_ignored: Any) -> bool:
        return self._root.delete(collection_name)

    def rename_collection(self, old_collection_name: str, new_collection_name: str) -> bool:
        # util/qdrant_manager.py:99 calls this; the upstream client has no such method, the drop-in does
        self._root.rename(old_collection_name, new_collection_name)
        return True

    # ------------------------------------------------------------------ points
    def count(self, collection_name: str, count_filter=None, exact: bool = True, **_ignored: Any) -> CountResult:
        col = self._root.get(collection_name)
        if count_filter is None:
            return CountResult(count=len(col))
        return CountResult(count=len(col.filter_slots(count_filter)))

    def upsert(self, collection_name: str, points, wait: bool = True, **_ignored: Any) -> UpdateResult:
        col = self._root.get(collection_name)
        if isinstance(points, Batch):
            vectors = np.asarray(points.vectors, dtype=np.float32)
            col.upsert_many(points.ids, vectors, points.payloads)
        else:
            for p in points:
                vec = p.vector
                if isinstance(vec, dict):
                    raise ValueError("named vectors are not supported by this drop-in")
                col.upsert(p.id, vec, p.payload)
        return UpdateResult(operation_id=0, status=UpdateStatus.COMPLETED)

    def upsert_embeddings(self, collection_name: str, ids, embeddings, payloads=None) -> UpdateResult:
        """Batched upsert of embeddings held in a torch CUDA tensor [n, dim] (e.g. ``model.encode_image(batch)``):
        the device-to-device counterpart of the per-image ``client.upsert`` at 31_…py:178-179 (§8 f3)."""
        col = self._root.get(collection_name)
        if hasattr(embeddings, "is_cuda") and embeddings.is_cuda:
            col.upsert_device(list(ids), embeddings, payloads)
        else:
            col.upsert_many(list(ids), np.asarray(embeddings, dtype=np.float32), payloads)
        return UpdateResult(operation_id=0, status=UpdateStatus.COMPLETED)

    def upload_collection(self, collection_name: str, vectors, payload=None, ids=None, **_ignored: Any) -> None:
        """Bulk path: vectors [n, dim] (numpy), ids default to 0..n-1 appended after existing ints."""
        col = self._root.get(collection_name)
        vectors = np.asarray(vectors, dtype=np.float32)
        n = vectors.shape[0]
        if ids is None:
            start = len(col)
            ids = range(start, start + n)
        col.upsert_many(list(ids), vectors, payload)

    def delete(self, collection_name: str, points_selector, wait: bool = True, **_ignored: Any) -> UpdateResult:
        col = self._root.get(collection_name)
        if hasattr(points_selector, "points"):
            ids = list(points_selector.points)
        elif hasattr(points_selector, "filter"):
            ids = [col.ids[s] for s in col.filter_slots(points_selector.filter) or []]
        elif hasattr(points_selector, "must") or hasattr(points_selector, "should"):
            ids = [col.ids[s] for s in col.filter_slots(points_selector) or []]
        else:
            ids = list(points_selector)
        col.delete(ids)
        return UpdateResult(operation_id=0, status=UpdateStatus.COMPLETED)

    def _records(self, col: Collection, slots: Sequence[int], with_payload, with_vectors) -> List[Record]:
        vecs = col.stored_vectors(slots) if with_vectors and len(slots) else None
        out = []
        for i, s in enumerate(slots):
            out.append(Record(id=col.ids[s], payload=dict(col.payloads[s]) if with_payload else None,
                              vector=vecs[i].tolist() if vecs is not None else None))
        return out

    def scroll(self, collection_name: str, scroll_filter=None, limit: int = 10, offset=None,
               with_payload=True, with_vectors=False, **_ignored: Any):
        """-> (records, next_page_offset); call sites 32_…py:78-82,123-131 and 33_…py:96-106,139-145."""
        col = self._root.get(collection_name)
        if limit is None or int(limit) < 1:
            raise ValueError("limit must be >= 1")
        slots, nxt = col.scroll(scroll_filter, int(limit), offset)
        return self._records(col, slots, bool(with_payload), bool(with_vectors)), nxt

    def retrieve(self, collection_name: str, ids: Iterable, with_payload=True, with_vectors=False,
                 **_ignored: Any) -> List[Record]:
        col = self._root.get(collection_name)
        slots = [col.slot_of[c] for c in (canonical_id(i) for i in ids) if c in col.slot_of]
        return self._records(col, slots, bool(with_payload), bool(with_vectors))

    # ------------------------------------------------------------------ search
    def _scored(self, col: Collection, scores, slots, with_payload, with_vectors, score_threshold,
                is_distance: Optional[bool] = None) -> List[ScoredPoint]:
        # EUCLID / MANHATTAN scores are distances (ascending, smaller = closer): the threshold is an upper bound
        if is_distance is None:
            is_distance = col.distance in ("Euclid", "Manhattan")
        keep = [(float(sc), int(s)) for sc, s in zip(scores, slots)
                if s >= 0 and (score_threshold is None
                               or (sc <= score_threshold if is_distance else sc >= score_threshold))]
        vecs = col.stored_vectors([s for _, s in keep]) if with_vectors and keep else None
        return [ScoredPoint(id=col.ids[s], version=0, score=sc,
                            payload=dict(col.payloads[s]) if with_payload else None,
                            vector=vecs[i].tolist() if vecs is not None else None)
                for i, (sc, s) in enumerate(keep)]

    def search(self, collection_name: str, query_vector, query_filter=None, limit: int = 10, offset: int = 0,
               with_payload=True, with_vectors=False, score_threshold: Optional[float] = None,
               **_ignored: Any) -> List[ScoredPoint]:
        col = self._root.get(collection_name)
        q = np.asarray(query_vector, dtype=np.float32).reshape(1, -1)
        if q.shape[1] != col.dim:
            raise ValueError(f"Wrong input: Vector dimension error: expected dim: {col.dim}, got {q.shape[1]}")
        k = int(limit) + int(offset or 0)
        if k < 1:
            return []
        scores, slots = col.search(q, k, query_filter)
        return self._scored(col, scores[0], slots[0], bool(with_payload), bool(with_vectors), score_threshold)[int(offset or 0):]

    def query_points(self, collection_name: str, query=None, query_filter=None, limit: int = 10, offset: int = 0,
                     with_payload=True, with_vectors=False, score_threshold: Optional[float] = None,
                     **_ignored: Any) -> QueryResponse:
        if isinstance(query, RecommendQuery):
            rec = query.recommend
            return QueryResponse(points=self.recommend(
                collection_name, rec.positive, rec.negative, query_filter, limit, offset, with_payload, with_vectors,
                score_threshold, _ignored.get("using"), _ignored.get("lookup_from"), rec.strategy))
        if isinstance(query, (DiscoverQuery, ContextQuery)):
            target, context = ((query.discover.target, query.discover.context) if isinstance(query, DiscoverQuery)
                               else (None, query.context))
            req = DiscoverRequest(target=target, context=context, filter=query_filter, limit=limit, offset=offset,
                                  with_payload=with_payload, with_vector=with_vectors, using=_ignored.get("using"),
                                  lookup_from=_ignored.get("lookup_from"))
            return QueryResponse(points=self._discover(collection_name, [req], score_threshold)[0])
        if isinstance(query, NearestQuery):
            req = QueryRequest(query=query, filter=query_filter, limit=limit, offset=offset, with_payload=with_payload,
                               with_vector=with_vectors, score_threshold=score_threshold, using=_ignored.get("using"),
                               lookup_from=_ignored.get("lookup_from"), prefetch=_ignored.get("prefetch"))
            if query.mmr is None:
                vec = self._nearest_vector(req)
                return QueryResponse(points=self.search(collection_name, vec, query_filter, limit, offset, with_payload,
                                                        with_vectors, score_threshold))
            return QueryResponse(points=self._mmr(collection_name, [req])[0])
        return QueryResponse(points=self.search(collection_name, query, query_filter, limit, offset, with_payload,
                                                with_vectors, score_threshold))

    @staticmethod
    def _nearest_vector(r):
        """The vector of a ``QueryRequest`` whose query is a ``NearestQuery``; what this drop-in does not support is a
        ValueError."""
        if r.using is not None:
            raise ValueError("query_points: named vectors (using=) are not supported by this drop-in")
        if r.lookup_from is not None:
            raise ValueError("query_points: lookup_from (vectors from another collection) is not supported")
        if r.prefetch is not None:
            raise ValueError("query_points: prefetch (and fusion) is not supported by this drop-in")
        v = r.query.nearest
        if isinstance(v, (str, uuid.UUID)) or (isinstance(v, (int, np.integer)) and not isinstance(v, bool)):
            raise ValueError("query_points: NearestQuery(nearest=<point id>) is not supported; pass the vector")
        return v

    def _mmr(self, collection_name: str, requests) -> List[List[ScoredPoint]]:
        """``QueryRequest``s whose query is a ``NearestQuery`` with ``mmr``: one device call (``Collection.search_mmr``)
        per distinct (limit + offset, candidates_limit)."""
        col = self._root.get(collection_name)
        plans = []
        for r in requests:
            q = np.asarray(self._nearest_vector(r), dtype=np.float32).reshape(-1)
            if q.shape[0] != col.dim:
                raise ValueError(f"Wrong input: Vector dimension error: expected dim: {col.dim}, got {q.shape[0]}")
            m = r.query.mmr
            k = int(r.limit) + int(r.offset or 0)
            div = 0.5 if m.diversity is None else float(m.diversity)
            if not 0.0 <= div <= 1.0:
                raise ValueError(f"query_points: mmr diversity must be in [0, 1], got {m.diversity!r}")
            cand = k if m.candidates_limit is None else int(m.candidates_limit)
            if cand < k:
                raise ValueError(f"query_points: mmr candidates_limit = {cand} is smaller than limit + offset = {k}")
            if cand > MAX_MMR_CANDIDATES:
                raise ValueError(f"query_points: mmr candidates_limit = {cand} exceeds {MAX_MMR_CANDIDATES}")
            plans.append((q, k, cand, div))
        out: List[List[ScoredPoint]] = [[] for _ in requests]
        groups: Dict[tuple, List[int]] = {}
        for i, (_, k, cand, _) in enumerate(plans):
            if k >= 1:
                groups.setdefault((k, cand), []).append(i)
        for (k, cand), members in groups.items():
            scores, slots = col.search_mmr(np.stack([plans[i][0] for i in members]), k, cand,
                                           np.array([plans[i][3] for i in members]),
                                           [requests[i].score_threshold for i in members],
                                           [requests[i].filter for i in members])
            for j, i in enumerate(members):
                r = requests[i]
                out[i] = self._scored(col, scores[j], slots[j], bool(r.with_payload), bool(r.with_vector),
                                      r.score_threshold)[int(r.offset or 0):]
        return out

    def query_batch_points(self, collection_name: str, requests, **_ignored: Any) -> List[QueryResponse]:
        """One ``query_points`` per ``QueryRequest``; each kind of query goes to its batch path: vectors and plain
        ``NearestQuery`` to ``search_batch``, ``NearestQuery`` with ``mmr`` to one device call per distinct (limit +
        offset, candidates_limit), ``RecommendQuery`` to ``recommend_batch``, ``DiscoverQuery`` / ``ContextQuery`` to
        discovery.  The output equals the per-request ``query_points`` loop."""
        requests = list(requests)
        out: List[List[ScoredPoint]] = [[] for _ in requests]
        kinds: Dict[str, List[int]] = {}
        for i, r in enumerate(requests):
            q = r.query
            kind = ("mmr" if isinstance(q, NearestQuery) and q.mmr is not None else "recommend"
                    if isinstance(q, RecommendQuery) else "discover" if isinstance(q, (DiscoverQuery, ContextQuery))
                    else "search")
            kinds.setdefault(kind, []).append(i)
        for kind, members in kinds.items():
            reqs = [requests[i] for i in members]
            if kind == "search":
                res = self.search_batch(collection_name, [SearchRequest(
                    vector=self._nearest_vector(r) if isinstance(r.query, NearestQuery) else r.query, filter=r.filter,
                    limit=r.limit, offset=r.offset, with_payload=r.with_payload, with_vector=r.with_vector,
                    score_threshold=r.score_threshold) for r in reqs])
            elif kind == "mmr":
                res = self._mmr(collection_name, reqs)
            elif kind == "recommend":
                res = self.recommend_batch(collection_name, [RecommendRequest(
                    positive=r.query.recommend.positive, negative=r.query.recommend.negative, filter=r.filter,
                    limit=r.limit, offset=r.offset, with_payload=r.with_payload, with_vector=r.with_vector,
                    score_threshold=r.score_threshold, using=r.using, lookup_from=r.lookup_from,
                    strategy=r.query.recommend.strategy) for r in reqs])
            else:
                res = [None] * len(reqs)
                by_thr: Dict[Any, List[int]] = {}
                for j, r in enumerate(reqs):
                    by_thr.setdefault(r.score_threshold, []).append(j)
                for thr, js in by_thr.items():
                    dreqs = []
                    for j in js:
                        r = reqs[j]
                        target, context = ((r.query.discover.target, r.query.discover.context)
                                           if isinstance(r.query, DiscoverQuery) else (None, r.query.context))
                        dreqs.append(DiscoverRequest(target=target, context=context, filter=r.filter, limit=r.limit,
                                                     offset=r.offset, with_payload=r.with_payload,
                                                     with_vector=r.with_vector, using=r.using,
                                                     lookup_from=r.lookup_from))
                    for j, pts in zip(js, self._discover(collection_name, dreqs, thr)):
                        res[j] = pts
            for i, pts in zip(members, res):
                out[i] = pts
        return [QueryResponse(points=p) for p in out]

    def search_batch(self, collection_name: str, requests=None, queries=None, k: Optional[int] = None,
                     row_filter=None, query_filters=None, **_ignored: Any):
        """Two forms: ``requests=[SearchRequest]`` -> list of ScoredPoint lists (upstream API), the same as one
        ``search`` per request; or the tensor form ``queries=[Q, dim], k=`` -> (scores [Q,k] float32, ids: list of Q
        lists), filtered by ``row_filter`` (every query) or ``query_filters`` (one filter or None per query)."""
        col = self._root.get(collection_name)
        if requests is not None:
            requests = list(requests)
            vecs = []
            for r in requests:
                q = np.asarray(r.vector, dtype=np.float32).reshape(1, -1)
                if q.shape[1] != col.dim:
                    raise ValueError(f"Wrong input: Vector dimension error: expected dim: {col.dim}, got {q.shape[1]}")
                vecs.append(q[0])
            # one device search per distinct limit + offset: a large limit does not drag the others to a larger k
            by_k: Dict[int, List[int]] = {}
            for i, r in enumerate(requests):
                by_k.setdefault(int(r.limit) + int(r.offset or 0), []).append(i)
            out: List[List[ScoredPoint]] = [[] for _ in requests]
            for kk, members in by_k.items():
                if kk < 1:
                    continue
                scores, slots = col.search(np.stack([vecs[i] for i in members]), kk,
                                           filters=[requests[i].filter for i in members])
                for j, i in enumerate(members):
                    r = requests[i]
                    out[i] = self._scored(col, scores[j], slots[j], bool(r.with_payload), bool(r.with_vector),
                                          r.score_threshold)[int(r.offset or 0):]
            return out
        if queries is None or k is None:
            raise ValueError("search_batch needs either requests= or queries= and k=")
        if row_filter is not None and query_filters is not None:
            raise ValueError("search_batch: pass row_filter (every query) or query_filters (one per query), not both")
        scores, slots = col.search(np.asarray(queries, dtype=np.float32), int(k), row_filter, filters=query_filters)
        id_of = np.asarray(col.ids + [None], dtype=object)          # slot -1 -> None through the last entry
        ids = id_of[np.asarray(slots)].tolist()
        return scores, ids

    # ------------------------------------------------------------------ recommendation (K6)
    def recommend(self, collection_name: str, positive=None, negative=None, query_filter=None, limit: int = 10,
                  offset: int = 0, with_payload=True, with_vectors=False, score_threshold: Optional[float] = None,
                  using=None, lookup_from=None, strategy=None, **_ignored: Any) -> List[ScoredPoint]:
        """Stored points like the ``positive`` examples and unlike the ``negative`` ones; each example is a point id
        (its stored vector) or a raw vector, 1 to 32 per request, and example points never appear in the answer.

        ``strategy`` (``RecommendStrategy`` or its string):
        * "average_vector" (default): a search of mean(positive), or 2 mean(positive) - mean(negative) when there are
          negatives, composed in float64 and rounded to float32 once.  Scores are the collection's search scores
          (distances for Euclid / Manhattan, where ``score_threshold`` is an upper bound).
        * "best_score": per stored row, bp / bn = its best search key against a positive / negative example, and the
          score is s(sim(bp)) if bp > bn, else -s(sim(bn)), with sim = identity (minus the L2 distance for Euclid) and
          s(y) = 0.5 (y / (1 + |y|) + 1).  This is the rule of Qdrant >= 1.7 as read from its source; it has not been
          checked against a live Qdrant.  Scores are larger-is-better for every distance: ``score_threshold`` keeps
          scores >= it.  Answered exactly by an fp64 sweep of the collection on the GPU.

        ``using`` (named vectors) and ``lookup_from`` (another collection) are not supported: ValueError."""
        req = RecommendRequest(positive=positive, negative=negative, filter=query_filter, limit=limit, offset=offset,
                               with_payload=with_payload, with_vector=with_vectors, score_threshold=score_threshold,
                               using=using, lookup_from=lookup_from, strategy=strategy)
        return self.recommend_batch(collection_name, [req])[0]

    def recommend_batch(self, collection_name: str, requests, **_ignored: Any) -> List[List[ScoredPoint]]:
        """One ``recommend`` per ``RecommendRequest``, answered with one device call per strategy and distinct
        limit + offset + example ids; the output equals the per-request loop."""
        col = self._root.get(collection_name)
        requests = list(requests)
        by_strategy: Dict[str, List[int]] = {}
        for i, r in enumerate(requests):
            if r.using is not None:
                raise ValueError("recommend: named vectors (using=) are not supported by this drop-in")
            if r.lookup_from is not None:
                raise ValueError("recommend: lookup_from (examples from another collection) is not supported")
            s = r.strategy.value if isinstance(r.strategy, RecommendStrategy) else (r.strategy or "average_vector")
            if s not in ("average_vector", "best_score"):
                raise ValueError(f"unknown recommend strategy {r.strategy!r}")
            by_strategy.setdefault(s, []).append(i)
        out: List[List[ScoredPoint]] = [[] for _ in requests]
        for s, members in by_strategy.items():
            res = col.recommend([(requests[i].positive, requests[i].negative, requests[i].filter,
                                  int(requests[i].limit) + int(requests[i].offset or 0)) for i in members], s)
            is_distance = s == "average_vector" and col.distance in ("Euclid", "Manhattan")
            for (scores, slots), i in zip(res, members):
                r = requests[i]
                out[i] = self._scored(col, scores, slots, bool(r.with_payload), bool(r.with_vector), r.score_threshold,
                                      is_distance)[int(r.offset or 0):]
        return out

    # ------------------------------------------------------------------ discovery and context search (K7)
    def discover(self, collection_name: str, target=None, context=None, query_filter=None, search_params=None,
                 limit: int = 10, offset: int = 0, with_payload=True, with_vectors=False, using=None,
                 lookup_from=None, **_ignored: Any) -> List[ScoredPoint]:
        """Stored points ranked by ``target`` within the region that ``context`` marks out.  ``context`` is a list of
        pairs, or one pair; a pair is a ``ContextExamplePair``, a ``ContextPair`` or a (positive, negative) tuple.
        Every example is a point id (its stored vector) or a raw vector, 1 to 32 per request (the target and two per
        pair), and example points never appear in the answer.

        With a pair's keys P / N (the collection's search key of a row against the positive / negative example), sim
        the identity (minus the L2 distance for Euclid), f(y) = y / (1 + |y|), s(y) = 0.5 (f(y) + 1) and MARGIN =
        2**-23, a row scores
        * with a target (discovery): the sum over pairs of (+1 if P > N else -1), plus s(sim(key of the target));
        * without (context search): the sum over pairs of f(min(sim(P) - sim(N) - MARGIN, 0)), which is 0 for every
          row on the positive side of every pair; ties are ordered by point slot.
        This is the rule of Qdrant >= 1.7 as read from its source; it has not been checked against a live Qdrant.
        Scores are larger-is-better for every distance.  Answered exactly by an fp64 sweep of the collection on the
        GPU.  A request with neither a target nor a context pair is a ValueError; ``using`` (named vectors) and
        ``lookup_from`` (another collection) are not supported: ValueError."""
        req = DiscoverRequest(target=target, context=context, filter=query_filter, params=search_params, limit=limit,
                              offset=offset, with_payload=with_payload, with_vector=with_vectors, using=using,
                              lookup_from=lookup_from)
        return self.discover_batch(collection_name, [req])[0]

    def discover_batch(self, collection_name: str, requests, **_ignored: Any) -> List[List[ScoredPoint]]:
        """One ``discover`` per ``DiscoverRequest``, answered with one device call per distinct limit + offset +
        example ids; the output equals the per-request loop."""
        return self._discover(collection_name, list(requests), None)

    def _discover(self, collection_name: str, requests, score_threshold) -> List[List[ScoredPoint]]:
        col = self._root.get(collection_name)
        plans = []
        for r in requests:
            if r.using is not None:
                raise ValueError("discover: named vectors (using=) are not supported by this drop-in")
            if r.lookup_from is not None:
                raise ValueError("discover: lookup_from (examples from another collection) is not supported")
            pairs = _context_pairs(r.context)
            if r.target is None and not pairs:
                raise ValueError("discover: a request needs a target or at least one context pair")
            plans.append((r.target, pairs, r.filter, int(r.limit) + int(r.offset or 0)))
        res = col.discover(plans)
        return [self._scored(col, scores, slots, bool(r.with_payload), bool(r.with_vector), score_threshold,
                             False)[int(r.offset or 0):]
                for (scores, slots), r in zip(res, requests)]

    # ------------------------------------------------------------------ delegates (K2)
    def build_delegates(self, collection_name: str, group_key: str = "class_name", scroll_filter=None,
                        kind: str = "average", alpha: float = 2.0):
        """Per-group delegate vectors of stored vectors in ONE segmented launch (K2 / K2b).

        The batched counterpart of the per-class loop in 32_create_delegate_vector.py:119-156: ``kind`` is
        "average" (compute_average :9-10), "centroid" (:12-15), "weighted" (:17-21, ``alpha``) or "medoid"
        (:23-26); the result is the stored (renormalised) form the script's upsert would leave.
        -> (group values, [G, dim] float32)."""
        col = self._root.get(collection_name)
        names, row_idx, offsets = col.group_rows(group_key, scroll_filter)
        col.flush()
        if kind == "average":
            return names, col.gallery.segment_mean(offsets, row_idx=row_idx)
        return names, col.gallery.segment_delegates(kind, offsets, row_idx=row_idx, alpha=alpha)[0]

    def close(self, **_ignored: Any) -> None:
        if self._key is None:
            self._root.close()
        else:
            for col in list(self._root.open_collections.values()):
                col.save()
