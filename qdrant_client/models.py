"""Model classes of the ``qdrant_client`` API subset the reference scripts use.

Plain Python objects with the constructor keywords and attributes of the third-party classes
(``qdrant_client.models`` / ``qdrant_client.http.models``): see SURVEY.md §8(b) and the call sites
util/qdrant_manager.py:2,61-66,82-85; 31_…py:20,178; 32_…py:6,104-117,125-129; 33_…py:13,98-137.
"""
from __future__ import annotations

import enum
from typing import Any, Dict, List, Optional, Sequence, Union


class Distance(str, enum.Enum):
    COSINE = "Cosine"
    EUCLID = "Euclid"
    DOT = "Dot"
    MANHATTAN = "Manhattan"


class _Model:
    """Keyword-only constructor + attribute access + value equality, like a pydantic model."""

    _fields: Sequence[str] = ()
    _defaults: Dict[str, Any] = {}
    _aliases: Dict[str, str] = {}

    def __init__(self, *args, **kwargs):
        if args:
            if len(args) > len(self._fields):
                raise TypeError(f"{type(self).__name__} takes at most {len(self._fields)} positional arguments")
            for name, value in zip(self._fields, args):
                if name in kwargs:
                    raise TypeError(f"{type(self).__name__}: multiple values for {name!r}")
                kwargs[name] = value
        for alias, name in self._aliases.items():
            if alias in kwargs:
                kwargs[name] = kwargs.pop(alias)
        unknown = set(kwargs) - set(self._fields)
        if unknown:
            raise TypeError(f"{type(self).__name__}: unexpected field(s) {sorted(unknown)}")
        for name in self._fields:
            if name in kwargs:
                setattr(self, name, kwargs[name])
            elif name in self._defaults:
                d = self._defaults[name]
                setattr(self, name, d() if callable(d) else d)
            else:
                raise TypeError(f"{type(self).__name__}: missing required field {name!r}")

    def dict(self) -> Dict[str, Any]:
        return {name: getattr(self, name) for name in self._fields}

    model_dump = dict

    def __eq__(self, other):
        return type(self) is type(other) and self.dict() == other.dict()

    def __repr__(self):
        return f"{type(self).__name__}({', '.join(f'{k}={getattr(self, k)!r}' for k in self._fields)})"


class VectorParams(_Model):
    _fields = ("size", "distance", "hnsw_config", "quantization_config", "on_disk", "datatype")
    _defaults = {"hnsw_config": None, "quantization_config": None, "on_disk": None, "datatype": None}


class PointStruct(_Model):
    _fields = ("id", "vector", "payload")
    _defaults = {"payload": None}


class Batch(_Model):
    _fields = ("ids", "vectors", "payloads")
    _defaults = {"payloads": None}


class MatchValue(_Model):
    _fields = ("value",)


class MatchAny(_Model):
    _fields = ("any",)


class MatchExcept(_Model):
    _fields = ("except_",)
    _aliases = {"except": "except_"}


class MatchText(_Model):
    _fields = ("text",)


class Range(_Model):
    _fields = ("lt", "gt", "gte", "lte")
    _defaults = {"lt": None, "gt": None, "gte": None, "lte": None}


class FieldCondition(_Model):
    _fields = ("key", "match", "range")
    _defaults = {"match": None, "range": None}


class HasIdCondition(_Model):
    _fields = ("has_id",)


class PayloadField(_Model):
    _fields = ("key",)


class IsNullCondition(_Model):
    _fields = ("is_null",)


class IsEmptyCondition(_Model):
    _fields = ("is_empty",)


class Filter(_Model):
    _fields = ("must", "should", "must_not")
    _defaults = {"must": None, "should": None, "must_not": None}


class SearchRequest(_Model):
    _fields = ("vector", "limit", "filter", "with_payload", "with_vector", "score_threshold", "offset")
    _defaults = {"filter": None, "with_payload": None, "with_vector": None, "score_threshold": None, "offset": 0}


class RecommendStrategy(str, enum.Enum):
    """average_vector (the default): one search of the composed vector; best_score: per row, the best positive against
    the best negative example (exact fp64 sweep on the device)."""
    AVERAGE_VECTOR = "average_vector"
    BEST_SCORE = "best_score"


class RecommendRequest(_Model):
    _fields = ("positive", "negative", "filter", "params", "limit", "offset", "with_payload", "with_vector",
               "score_threshold", "using", "lookup_from", "strategy", "shard_key")
    _defaults = {"positive": None, "negative": None, "filter": None, "params": None, "offset": 0, "with_payload": None,
                 "with_vector": None, "score_threshold": None, "using": None, "lookup_from": None, "strategy": None,
                 "shard_key": None}


class RecommendInput(_Model):
    _fields = ("positive", "negative", "strategy")
    _defaults = {"positive": None, "negative": None, "strategy": None}


class RecommendQuery(_Model):
    _fields = ("recommend",)


class ContextExamplePair(_Model):
    """One correction of ``discover``: stored points should be like ``positive`` and unlike ``negative`` (each a point
    id or a vector)."""
    _fields = ("positive", "negative")


class DiscoverRequest(_Model):
    _fields = ("target", "context", "filter", "params", "limit", "offset", "with_payload", "with_vector", "using",
               "lookup_from", "shard_key")
    _defaults = {"target": None, "context": None, "filter": None, "params": None, "offset": 0, "with_payload": None,
                 "with_vector": None, "using": None, "lookup_from": None, "shard_key": None}


class ContextPair(_Model):
    """A (positive, negative) pair of the query API (``DiscoverInput.context``, ``ContextQuery.context``)."""
    _fields = ("positive", "negative")


class DiscoverInput(_Model):
    _fields = ("target", "context")


class DiscoverQuery(_Model):
    _fields = ("discover",)


class ContextQuery(_Model):
    """Context search: ``context`` is one ``ContextPair`` or a list of them."""
    _fields = ("context",)


class Mmr(_Model):
    """Maximal marginal relevance of a ``NearestQuery``: ``limit`` picks among the exact top-``candidates_limit``, each
    trading relevance against similarity to the points already picked.  Defaults of this drop-in (not checked against
    Qdrant): ``diversity`` 0.5, ``candidates_limit`` = limit + offset."""
    _fields = ("diversity", "candidates_limit")
    _defaults = {"diversity": None, "candidates_limit": None}


class NearestQuery(_Model):
    """Nearest-neighbour search of the query API: ``nearest`` is a vector; with ``mmr`` the answer is diversified."""
    _fields = ("nearest", "mmr")
    _defaults = {"mmr": None}


class QueryRequest(_Model):
    """One request of ``query_batch_points``: ``query`` is a vector, a ``NearestQuery``, a ``RecommendQuery``, a
    ``DiscoverQuery`` or a ``ContextQuery``."""
    _fields = ("query", "filter", "limit", "offset", "with_payload", "with_vector", "score_threshold", "using",
               "lookup_from", "prefetch", "params", "shard_key")
    _defaults = {"query": None, "filter": None, "limit": 10, "offset": 0, "with_payload": None, "with_vector": None,
                 "score_threshold": None, "using": None, "lookup_from": None, "prefetch": None, "params": None,
                 "shard_key": None}


class PointIdsList(_Model):
    _fields = ("points",)


class FilterSelector(_Model):
    _fields = ("filter",)


# ---- results --------------------------------------------------------------------------------
class Record(_Model):
    _fields = ("id", "payload", "vector", "shard_key", "order_value")
    _defaults = {"payload": None, "vector": None, "shard_key": None, "order_value": None}


class ScoredPoint(_Model):
    _fields = ("id", "version", "score", "payload", "vector", "shard_key", "order_value")
    _defaults = {"version": 0, "payload": None, "vector": None, "shard_key": None, "order_value": None}


class QueryResponse(_Model):
    _fields = ("points",)


class UpdateStatus(str, enum.Enum):
    ACKNOWLEDGED = "acknowledged"
    COMPLETED = "completed"


class UpdateResult(_Model):
    _fields = ("operation_id", "status")
    _defaults = {"operation_id": 0, "status": UpdateStatus.COMPLETED}


class CountResult(_Model):
    _fields = ("count",)


class CollectionDescription(_Model):
    _fields = ("name",)


class CollectionsResponse(_Model):
    _fields = ("collections",)


class CollectionStatus(str, enum.Enum):
    GREEN = "green"
    YELLOW = "yellow"
    RED = "red"


class CollectionParams(_Model):
    _fields = ("vectors",)


class CollectionConfig(_Model):
    _fields = ("params",)


class CollectionInfo(_Model):
    _fields = ("status", "points_count", "vectors_count", "indexed_vectors_count", "segments_count", "config",
               "payload_schema")
    _defaults = {"status": CollectionStatus.GREEN, "vectors_count": None, "indexed_vectors_count": 0,
                 "segments_count": 1, "config": None, "payload_schema": dict}


PointId = Union[int, str]
Payload = Dict[str, Any]
VectorStruct = List[float]
