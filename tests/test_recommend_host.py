"""Host side of recommendation: ``recommend`` / ``recommend_batch`` / ``query_points(query=RecommendQuery(...))`` resolve
example ids to stored vectors, drop the example points from the answers, apply offset and score_threshold, compose the
average_vector query and group requests into device calls.  The gallery is a test double that answers ``recommend``
with the fp64 oracle (the device side is in tests/test_gpu_recommend.py)."""
from types import SimpleNamespace

import numpy as np
import pytest

from fakes import fake_gallery
from oracle import oracle_np as O
from oracle import oracle_reco as OR


class RecoFakeGallery(fake_gallery.FakeGallery):
    def search(self, queries, k, row_mask=None, want_scores64=False, out=None, stream=None, mask_of_query=None):
        if mask_of_query is None:
            return super().search(queries, k, row_mask, want_scores64, out, stream)
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        ids = np.asarray(mask_of_query, dtype=np.int32)
        masks = np.asarray(row_mask, dtype=np.uint32).reshape(-1, (len(self._rows) + 31) // 32)
        self.calls.append(("search_masks", len(q), k, len(masks)))
        scores = np.empty((len(q), k), dtype=np.float32)
        rows = np.empty((len(q), k), dtype=np.int64)
        for i in range(len(q)):
            one = fake_gallery.FakeGallery.search(self, q[i:i + 1], k, None if ids[i] < 0 else masks[ids[i]])
            self.calls.pop()
            scores[i], rows[i] = one.scores[0], one.rows[0]
        return SimpleNamespace(scores=scores, rows=rows, scores64=scores.astype(np.float64), stats={})

    def recommend(self, examples, signs, offsets, k, row_mask=None, mask_of_request=None, want_keys=False):
        ex = np.asarray(examples, dtype=np.float32).reshape(-1, self.dim)
        signs, offsets = np.asarray(signs, dtype=np.int8), np.asarray(offsets, dtype=np.int64)
        R, n = len(offsets) - 1, len(self._rows)
        assert len(signs) == len(ex) == offsets[-1] and offsets[0] == 0 and np.all(np.diff(offsets) >= 1)
        assert np.all(np.diff(offsets) <= 32) and set(signs.tolist()) <= {1, -1} and 1 <= k <= 1024
        if row_mask is None:
            allowed, n_masks = None, 0
        else:
            masks = np.asarray(row_mask, dtype=np.uint32).reshape(-1, (n + 31) // 32)
            ids = np.zeros(R, dtype=np.int32) if mask_of_request is None else np.asarray(mask_of_request)
            allowed = [None if i < 0 else O.unpack_row_mask(masks[i], n) for i in ids]
            n_masks = len(masks)
        self.calls.append(("recommend", R, k, n_masks))
        s, i = OR.recommend_topk(ex, signs, offsets, self._rows, k, self.metric, allowed)
        return SimpleNamespace(scores=s.astype(np.float32), rows=i, scores64=s if want_keys else None, stats={})


@pytest.fixture()
def client(store_dir, monkeypatch):
    import retrieval_based_object_detection_b200 as pkg
    import retrieval_based_object_detection_b200.gallery as gallery

    monkeypatch.setattr(gallery, "Gallery", RecoFakeGallery)
    monkeypatch.setattr(pkg, "Gallery", RecoFakeGallery)
    from qdrant_client import QdrantClient

    return QdrantClient(host="localhost", port=6333)


def _fill(client, distance="COSINE", n=300, dim=16):
    from qdrant_client import models

    client.recreate_collection("r", vectors_config=models.VectorParams(size=dim, distance=getattr(models.Distance, distance)))
    rng = np.random.default_rng(5)
    vecs = rng.standard_normal((n, dim)).astype(np.float32)
    client.upsert("r", points=models.Batch(ids=list(range(n)), vectors=vecs.tolist(),
                                           payloads=[{"class_name": f"c{i % 7}"} for i in range(n)]))
    col = client._root.get("r")
    return col, col.stored_vectors(range(n))


def _cls(j):
    from qdrant_client import models

    return models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value=f"c{j}"))])


def _pairs(points):
    return [(p.id, p.score) for p in points]


@pytest.mark.parametrize("distance", ["COSINE", "EUCLID"])
def test_best_score_with_ids_and_vectors_matches_the_oracle(client, distance):
    col, stored = _fill(client, distance)
    metric = distance.lower()
    rng = np.random.default_rng(6)
    raw = rng.standard_normal((2, 16)).astype(np.float32)
    pos, neg = [3, raw[0].tolist()], [17, 40, raw[1].tolist()]
    got = client.recommend("r", positive=pos, negative=neg, limit=12, strategy="best_score")
    ex = np.stack([stored[3], raw[0], stored[17], stored[40], raw[1]])
    s, i = OR.recommend_topk(ex, [1, 1, -1, -1, -1], [0, 5], stored, 15, metric)
    keep = ~np.isin(i[0], [3, 17, 40])
    assert [p.id for p in got] == i[0][keep][:12].tolist()
    assert np.allclose([p.score for p in got], s[0][keep][:12].astype(np.float32), rtol=0, atol=0)
    assert all(p.payload == {"class_name": f"c{p.id % 7}"} for p in got)
    # positives only, negatives only: each branch of the rule alone
    for kw in ({"positive": [5]}, {"negative": [5, 6]}):
        got = client.recommend("r", limit=4, strategy=models_strategy("best_score"), **kw)
        P, Nn = kw.get("positive", []), kw.get("negative", [])
        s, i = OR.recommend_topk(stored[P + Nn], [1] * len(P) + [-1] * len(Nn), [0, len(P) + len(Nn)], stored,
                                 4 + len(P) + len(Nn), metric)
        keep = ~np.isin(i[0], P + Nn)
        assert [p.id for p in got] == i[0][keep][:4].tolist()
        assert all(p.score < 0 for p in got) == (not P)


def models_strategy(name):
    from qdrant_client import models

    return models.RecommendStrategy(name)


def test_example_ids_never_appear_even_inside_the_top_k(client):
    col, stored = _fill(client)
    g = col._ensure_gallery()
    for strategy in ("best_score", "average_vector"):
        # the stored rows of positives 10 and 11 are the two best hits of a search without the exclusion
        raw = g.recommend(stored[[10, 11]], [1, 1], [0, 2], 5) if strategy == "best_score" else \
            g.search(stored[[10, 11]].astype(np.float64).mean(axis=0, keepdims=True).astype(np.float32), 5)
        assert {10, 11} & set(np.asarray(raw.rows[0]).tolist())
        got = client.recommend("r", positive=[10, 11], limit=5, strategy=strategy)
        assert len(got) == 5 and not {10, 11} & {p.id for p in got}
        # an id given twice is fetched once
        g.calls.clear()
        client.recommend("r", positive=[10, 10, 11], limit=5, strategy=strategy)
        assert [c[2] for c in g.calls if c[0] in ("recommend", "search")] == [7]


def test_unknown_id_names_it(client):
    _fill(client)
    with pytest.raises(ValueError, match="point 999 not found in collection 'r'"):
        client.recommend("r", positive=[1, 999], strategy="best_score")
    with pytest.raises(ValueError, match="12345678-1234-5678-1234-567812345678"):
        client.recommend("r", positive=[1], negative=["12345678-1234-5678-1234-567812345678"])


@pytest.mark.parametrize("strategy", ["best_score", "average_vector"])
@pytest.mark.parametrize("distance", ["COSINE", "MANHATTAN"])
def test_offset_and_score_threshold(client, strategy, distance):
    _fill(client, distance)
    full = client.recommend("r", positive=[1, 2], negative=[3], limit=20, strategy=strategy)
    assert client.recommend("r", positive=[1, 2], negative=[3], limit=5, offset=3, strategy=strategy) == full[3:8]
    thr = full[9].score
    got = client.recommend("r", positive=[1, 2], negative=[3], limit=20, score_threshold=thr, strategy=strategy)
    # best_score is larger-is-better for every distance; average_vector keeps the collection's search scores
    if strategy == "average_vector" and distance == "MANHATTAN":
        want = [p for p in full if p.score <= thr]
    else:
        want = [p for p in full if p.score >= thr]
    assert got == want and len(got) >= 10


@pytest.mark.parametrize("distance", ["COSINE", "EUCLID"])
def test_average_vector_is_the_search_of_the_composed_vector(client, distance):
    col, stored = _fill(client, distance)
    raw = np.linspace(-1, 1, 16).astype(np.float32)
    for pos, neg in (([4, 9], []), ([4, raw.tolist()], [30, 31, 32])):
        P = [stored[x] if isinstance(x, int) else np.asarray(x, np.float32) for x in pos]
        Nn = [stored[x] for x in neg]
        q = np.mean(np.asarray(P, np.float64), axis=0)
        if Nn:
            q = 2 * q - np.mean(np.asarray(Nn, np.float64), axis=0)
        ex_ids = [x for x in pos + neg if isinstance(x, int)]
        want = [p for p in client.search("r", q.astype(np.float32), limit=8 + len(ex_ids)) if p.id not in ex_ids][:8]
        assert client.recommend("r", positive=pos, negative=neg, limit=8) == want
        assert client.recommend("r", positive=pos, negative=neg, limit=8, strategy="average_vector") == want


def test_recommend_batch_equals_the_loop_with_one_call_per_strategy_and_fetch(client):
    from qdrant_client import models

    col, stored = _fill(client)
    rng = np.random.default_rng(8)
    flts = [None, _cls(0), _cls(1), _cls(0), None, _cls(2)]
    reqs = []
    for i in range(24):
        pos = [int(x) for x in rng.choice(300, 1 + i % 3, replace=False)]
        neg = [int(x) for x in rng.choice(300, i % 2, replace=False)]
        if i % 5 == 0:
            neg.append(rng.standard_normal(16).tolist())
        reqs.append(models.RecommendRequest(positive=pos, negative=neg, filter=flts[i % len(flts)], limit=(3, 6)[i % 2],
                                            offset=i % 3, with_payload=i % 4 != 0, with_vector=i % 7 == 0,
                                            score_threshold=-0.5 if i % 6 == 0 else None,
                                            strategy=("best_score", models.RecommendStrategy.AVERAGE_VECTOR, None)[i % 3]))
    g = col._ensure_gallery()
    g.calls.clear()
    got = client.recommend_batch("r", reqs)
    calls = [c for c in g.calls if c[0] in ("recommend", "search", "search_masks")]
    want = [client.recommend("r", r.positive, r.negative, r.filter, r.limit, r.offset, bool(r.with_payload),
                             bool(r.with_vector), r.score_threshold, strategy=r.strategy) for r in reqs]
    assert got == want and all(len(p) > 0 for p in got)
    fetch = {}
    for r in reqs:
        s = "best_score" if r.strategy == "best_score" else "average_vector"
        n_ids = len({x for x in r.positive + r.negative if isinstance(x, int)})
        fetch.setdefault((s, r.limit + r.offset + n_ids), []).append(r)
    assert len(calls) == len(fetch)
    for c in calls:
        kind = "best_score" if c[0] == "recommend" else "average_vector"
        members = fetch[(kind, c[2])]
        assert c[1] == len(members)
        n_filters = len({repr(r.filter) for r in members if r.filter is not None})
        assert (c[3] if c[0] != "search" else 0) == n_filters


def test_recommend_query_form(client):
    from qdrant_client import models
    from qdrant_client.http import models as http_models

    _fill(client)
    assert http_models.RecommendQuery is models.RecommendQuery
    q = models.RecommendQuery(recommend=models.RecommendInput(positive=[1, 2], negative=[3], strategy="best_score"))
    got = client.query_points("r", query=q, query_filter=_cls(1), limit=4, offset=1).points
    assert got == client.recommend("r", [1, 2], [3], _cls(1), 4, 1, strategy="best_score")
    assert all(p.payload["class_name"] == "c1" for p in got) and len(got) == 4
    with pytest.raises(ValueError, match="named vectors"):
        client.query_points("r", query=q, using="image")


def test_limits_and_unsupported_arguments(client):
    _fill(client)
    client.recommend("r", positive=list(range(20)), negative=list(range(20, 32)), strategy="best_score")
    with pytest.raises(ValueError, match="1 to 32 examples, got 33"):
        client.recommend("r", positive=list(range(20)), negative=list(range(20, 33)), strategy="best_score")
    with pytest.raises(ValueError, match="1 to 32 examples, got 0"):
        client.recommend("r", positive=[], strategy="best_score")
    with pytest.raises(ValueError, match="needs at least one positive"):
        client.recommend("r", negative=[1])
    client.recommend("r", positive=[1, 2], limit=1020, offset=2, strategy="best_score")
    with pytest.raises(ValueError, match="1025 exceeds 1024"):
        client.recommend("r", positive=[1, 2], limit=1020, offset=3, strategy="best_score")
    with pytest.raises(ValueError, match="named vectors"):
        client.recommend("r", positive=[1], using="image")
    with pytest.raises(ValueError, match="lookup_from"):
        client.recommend("r", positive=[1], lookup_from={"collection": "other"})
    with pytest.raises(ValueError, match="unknown recommend strategy"):
        client.recommend("r", positive=[1], strategy="sum_scores")
    with pytest.raises(ValueError) as single:
        client.search("r", [0.1] * 15, limit=3)
    with pytest.raises(ValueError) as reco:
        client.recommend("r", positive=[1, [0.1] * 15], strategy="best_score")
    assert str(reco.value) == str(single.value)
    assert client.recommend("r", positive=[1], limit=0) == []
