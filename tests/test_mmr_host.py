"""Maximal marginal relevance on the host: the oracle's rule on hand-built 2-D cases whose answers are known by
construction, a seeded "augmented" gallery, and the client (``query_points(query=NearestQuery(mmr=Mmr(...)))`` and
``query_batch_points``) over a gallery test double that answers ``search_mmr`` with the fp64 oracle (the device side is
in tests/test_gpu_mmr.py)."""
from types import SimpleNamespace

import numpy as np
import pytest

from fakes import fake_gallery
from oracle import oracle_discover as OD
from oracle import oracle_mmr as OM
from oracle import oracle_np as O
from oracle import oracle_reco as OR


# ---------------------------------------------------------------------------------------------- the rule
def _pick(query, stored, limit, L, diversity, metric="dot"):
    return OM.mmr_select(np.asarray(query, np.float32), np.asarray(stored, np.float32), limit, L, diversity, metric)[0]


def test_the_first_pick_is_the_best_candidate_and_diversity_0_is_plain_search():
    stored = [[1.0, 0.0], [0.99, 0.1], [0.98, 0.12], [0.0, 0.9], [0.5, 0.5]]
    q = [1.0, 0.0]
    keys = OR.example_keys(np.asarray([q], np.float32), np.asarray(stored, np.float32), "dot")
    _, order = O.topk_from_scores(keys, 5)
    for d in (0.0, 0.3, 0.7, 1.0):
        assert _pick(q, stored, 3, 5, d)[0] == order[0][0]
    assert _pick(q, stored, 4, 5, 0.0).tolist() == order[0][:4].tolist()


def test_lambda_trades_relevance_against_similarity():
    # two near-copies of the best row and one less relevant but different row (DOT)
    stored = [[1.0, 0.0], [0.95, 0.0], [0.0, 0.8]]
    q = [1.0, 0.2]
    # relevance: 1.0, 0.95, 0.16.  After picking row 0: sim(row 0, row 1) = 0.95, sim(row 0, row 2) = 0
    # mmr(1) = lam 0.95 - d 0.95, mmr(2) = lam 0.16: row 2 wins once d > 0.79 / 1.74
    assert _pick(q, stored, 2, 3, 0.3).tolist() == [0, 1]
    assert _pick(q, stored, 2, 3, 0.5).tolist() == [0, 2]
    assert _pick(q, stored, 2, 3, 1.0).tolist() == [0, 2]


def test_diversity_1_ignores_relevance_after_the_first_pick():
    # COSINE: after row 0 every pick minimises its largest similarity to the picks, whatever its relevance
    stored = np.array([[1, 0], [0.8, 0.6], [0, 1], [-1, 0.05]], np.float32)
    assert _pick([1, 0.01], stored, 3, 4, 1.0, "cosine").tolist() == [0, 3, 2]


def test_exact_ties_go_to_the_smaller_candidate_rank():
    # rows 1 and 2 are mirror images: equal relevance is broken by row (rank), and after the first pick equal mmr too
    stored = np.array([[2, 0], [1, 1], [1, -1], [1, 1]], np.float32)
    assert _pick([1, 0], stored, 4, 4, 0.0).tolist() == [0, 1, 2, 3]
    # every later pick ties too (sim 2 to row 0 for all): the smaller rank wins each time
    assert _pick([1, 0], stored, 4, 4, 0.5).tolist() == [0, 1, 2, 3]
    # COSINE, rows 1 and 2 identical, row 3 their mirror image: all three tie after row 0, row 1 wins by rank, and then
    # its duplicate row 2 is penalised by sim(1, 2) = 1 while the mirror is not
    stored = np.array([[1, 0], [0.6, 0.8], [0.6, 0.8], [0.6, -0.8]], np.float32)
    assert _pick([1, 0], stored, 3, 4, 0.5, "cosine").tolist() == [0, 1, 3]
    assert _pick([1, 0], stored, 3, 4, 0.0, "cosine").tolist() == [0, 1, 2]


def test_euclid_uses_minus_the_distance_as_sim():
    stored = np.array([[0, 0], [0.1, 0], [3, 0]], np.float32)
    rows, keys = OM.mmr_select(np.array([0.0, 0.0], np.float32), stored, 2, 3, 0.5, "euclid")
    # rel = (0, -0.1, -3); after row 0: mmr(1) = 0.5 (-0.1) - 0.5 (-0.1) = 0, mmr(2) = 0.5 (-3) - 0.5 (-3) = 0: a tie
    assert rows.tolist() == [0, 1]
    assert keys.tolist() == [0.0, -np.float64(np.float32(0.1)) ** 2]


def _augmented(n_src=40, copies=18, dim=32, seed=0):
    """Sources x noisy copies (like the reference's augmentation): row i is a copy of source i // copies."""
    rng = np.random.default_rng(seed)
    src = rng.standard_normal((n_src, dim)).astype(np.float32)
    x = np.repeat(src, copies, axis=0) + 0.05 * rng.standard_normal((n_src * copies, dim)).astype(np.float32)
    return O.l2_normalize_store(x, "f32")[0], src, copies


def test_mmr_returns_more_distinct_sources_than_plain_search():
    stored, src, copies = _augmented()
    rng = np.random.default_rng(1)
    for t in range(5):
        q = (src[t] + 0.6 * src[t + 1] + 0.5 * rng.standard_normal(src.shape[1])).astype(np.float32)
        plain = _pick(q, stored, 10, 10, 0.0, "cosine")
        mmr = _pick(q, stored, 10, 200, 0.5, "cosine")
        assert len(set(mmr // copies)) > len(set(plain // copies)) and len(set(plain // copies)) <= 2


# ---------------------------------------------------------------------------------------------- the client
class MmrFakeGallery(fake_gallery.FakeGallery):
    def _allowed(self, row_mask, mask_of_query, Q):
        n = len(self._rows)
        if row_mask is None:
            return [None] * Q, 0
        masks = np.asarray(row_mask, dtype=np.uint32).reshape(-1, (n + 31) // 32)
        ids = np.zeros(Q, dtype=np.int32) if mask_of_query is None else np.asarray(mask_of_query)
        return [None if i < 0 else O.unpack_row_mask(masks[i], n) for i in ids], len(masks)

    def search(self, queries, k, row_mask=None, want_scores64=False, out=None, stream=None, mask_of_query=None):
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        allowed, n_masks = self._allowed(row_mask, mask_of_query, len(q))
        self.calls.append(("search", len(q), k, n_masks))
        keys = OR.example_keys(q, self._rows, self.metric)
        s = np.full((len(q), k), -np.inf)
        i = np.full((len(q), k), -1, dtype=np.int64)
        for j in range(len(q)):
            s[j:j + 1], i[j:j + 1] = O.topk_from_scores(keys[j:j + 1], k, row_mask=allowed[j])
        return SimpleNamespace(scores=OM.user_scores(s, self.metric), rows=i, scores64=s, stats={})

    def search_mmr(self, queries, limit, candidates, diversity, score_threshold=None, row_mask=None,
                   mask_of_query=None, want_keys=False):
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        Q = len(q)
        assert 1 <= limit <= candidates <= 1024
        div = np.broadcast_to(np.asarray(diversity, np.float64), (Q,))
        thr = None if score_threshold is None else np.broadcast_to(np.asarray(score_threshold, np.float32), (Q,))
        assert np.all((div >= 0) & (div <= 1))
        allowed, n_masks = self._allowed(row_mask, mask_of_query, Q)
        self.calls.append(("search_mmr", Q, limit, candidates, n_masks))
        rows = np.full((Q, limit), -1, dtype=np.int64)
        keys = np.full((Q, limit), -np.inf)
        for j in range(Q):
            rows[j], keys[j] = OM.mmr_select(q[j], self._rows, limit, candidates, float(div[j]), self.metric,
                                             allowed[j], None if thr is None else float(thr[j]))
        scores = OM.user_scores(keys, self.metric)
        if self.metric in ("euclid", "manhattan"):
            scores[rows < 0] = np.inf
        return SimpleNamespace(scores=scores, rows=rows, scores64=keys if want_keys else None, stats={})

    def recommend(self, examples, signs, offsets, k, row_mask=None, mask_of_request=None, want_keys=False):
        offsets = np.asarray(offsets, dtype=np.int64)
        allowed, n_masks = self._allowed(row_mask, mask_of_request, len(offsets) - 1)
        self.calls.append(("recommend", len(offsets) - 1, k, n_masks))
        s, i = OR.recommend_topk(examples, signs, offsets, self._rows, k, self.metric, allowed)
        return SimpleNamespace(scores=s.astype(np.float32), rows=i, scores64=s, stats={})

    def discover(self, examples, roles, offsets, k, row_mask=None, mask_of_request=None, want_keys=False):
        offsets = np.asarray(offsets, dtype=np.int64)
        allowed, n_masks = self._allowed(row_mask, mask_of_request, len(offsets) - 1)
        self.calls.append(("discover", len(offsets) - 1, k, n_masks))
        s, i = OD.discover_topk(examples, roles, offsets, self._rows, k, self.metric, allowed)
        return SimpleNamespace(scores=s.astype(np.float32), rows=i, scores64=s, stats={})


@pytest.fixture()
def client(store_dir, monkeypatch):
    import retrieval_based_object_detection_b200 as pkg
    import retrieval_based_object_detection_b200.gallery as gallery

    monkeypatch.setattr(gallery, "Gallery", MmrFakeGallery)
    monkeypatch.setattr(pkg, "Gallery", MmrFakeGallery)
    from qdrant_client import QdrantClient

    return QdrantClient(host="localhost", port=6333)


def _fill(client, distance="COSINE", n=300, dim=16, augmented=False):
    from qdrant_client import models

    client.recreate_collection("m", vectors_config=models.VectorParams(size=dim, distance=getattr(models.Distance, distance)))
    rng = np.random.default_rng(5)
    if augmented:
        src = rng.standard_normal((n // 15, dim)).astype(np.float32)
        vecs = np.repeat(src, 15, axis=0) + 0.05 * rng.standard_normal((n // 15 * 15, dim)).astype(np.float32)
    else:
        vecs = rng.standard_normal((n, dim)).astype(np.float32)
    client.upsert("m", points=models.Batch(ids=list(range(len(vecs))), vectors=vecs.tolist(),
                                           payloads=[{"class_name": f"c{i % 7}"} for i in range(len(vecs))]))
    col = client._root.get("m")
    return col, col.stored_vectors(range(len(vecs)))


def _cls(j):
    from qdrant_client import models

    return models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value=f"c{j}"))])


def _mmr_q(v, diversity=None, candidates=None):
    from qdrant_client import models

    return models.NearestQuery(nearest=list(map(float, v)), mmr=models.Mmr(diversity=diversity, candidates_limit=candidates))


@pytest.mark.parametrize("distance", ["COSINE", "DOT", "EUCLID", "MANHATTAN"])
def test_query_points_matches_the_oracle_in_selection_order(client, distance):
    col, stored = _fill(client, distance, augmented=True)
    metric = distance.lower()
    q = stored[33] + 0.1
    got = client.query_points("m", query=_mmr_q(q, 0.6, 60), limit=8).points
    rows, keys = OM.mmr_select(q.astype(np.float32), stored, 8, 60, 0.6, metric)
    assert [p.id for p in got] == rows.tolist()
    assert [p.score for p in got] == OM.user_scores(keys, metric).tolist()
    assert all(p.payload == {"class_name": f"c{p.id % 7}"} for p in got)
    plain = client.search("m", q, limit=8)
    assert len({p.id // 15 for p in got}) > len({p.id // 15 for p in plain})


def test_client_defaults_offset_and_plain_nearest(client):
    from qdrant_client import models

    col, stored = _fill(client)
    q = stored[4] + 0.2
    g = col._ensure_gallery()
    g.calls.clear()
    got = client.query_points("m", query=_mmr_q(q), limit=5, offset=2).points
    # diversity 0.5, candidates_limit = limit + offset
    assert g.calls == [("search_mmr", 1, 7, 7, 0)]
    rows, _ = OM.mmr_select(q.astype(np.float32), stored, 7, 7, 0.5, "cosine")
    assert [p.id for p in got] == rows[2:].tolist()
    # without mmr a NearestQuery is the ordinary search
    assert (client.query_points("m", query=models.NearestQuery(nearest=q.tolist()), limit=5, offset=2).points
            == client.search("m", q, limit=5, offset=2))
    # diversity 0 is plain search, for any candidates_limit
    assert ([p.id for p in client.query_points("m", query=_mmr_q(q, 0.0, 300), limit=9).points]
            == [p.id for p in client.search("m", q, limit=9)])
    assert client.query_points("m", query=_mmr_q(q, 0.5, 10), limit=0).points == []


@pytest.mark.parametrize("distance", ["COSINE", "EUCLID"])
def test_score_threshold_restricts_the_candidates(client, distance):
    col, stored = _fill(client, distance)
    q = stored[7] + 0.05
    plain = client.search("m", q, limit=40)
    thr = plain[19].score
    got = client.query_points("m", query=_mmr_q(q, 0.9, 100), limit=10, score_threshold=thr).points
    # the request still fills its limit from the 20 candidates that pass, all within the threshold
    assert len(got) == 10 and {p.id for p in got} <= {p.id for p in plain[:20]}
    rows, _ = OM.mmr_select(q.astype(np.float32), stored, 10, 100, 0.9, distance.lower(), score_threshold=thr)
    assert [p.id for p in got] == rows.tolist()
    # fewer candidates than the limit: the answer is short
    thr = plain[3].score
    assert len(client.query_points("m", query=_mmr_q(q, 0.9, 100), limit=10, score_threshold=thr).points) == 4


def test_value_errors(client):
    from qdrant_client import models

    col, stored = _fill(client)
    q = stored[1].tolist()
    with pytest.raises(ValueError, match="candidates_limit = 9 is smaller than limit \\+ offset = 10"):
        client.query_points("m", query=_mmr_q(q, 0.5, 9), limit=8, offset=2)
    with pytest.raises(ValueError, match="candidates_limit = 1025 exceeds 1024"):
        client.query_points("m", query=_mmr_q(q, 0.5, 1025), limit=8)
    client.query_points("m", query=_mmr_q(q, 0.5, 1024), limit=8)
    for d in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError, match="diversity must be in \\[0, 1\\]"):
            client.query_points("m", query=_mmr_q(q, d), limit=8)
    with pytest.raises(ValueError, match="point id"):
        client.query_points("m", query=models.NearestQuery(nearest=3, mmr=models.Mmr(diversity=0.5)))
    with pytest.raises(ValueError, match="point id"):
        client.query_points("m", query=models.NearestQuery(nearest=3))
    with pytest.raises(ValueError, match="prefetch"):
        client.query_points("m", query=_mmr_q(q), prefetch=[{"query": q}])
    with pytest.raises(ValueError, match="named vectors"):
        client.query_points("m", query=_mmr_q(q), using="image")
    with pytest.raises(ValueError, match="lookup_from"):
        client.query_points("m", query=models.NearestQuery(nearest=q), lookup_from={"collection": "other"})
    with pytest.raises(ValueError) as single:
        client.search("m", q[:15], limit=3)
    with pytest.raises(ValueError) as mmr:
        client.query_points("m", query=_mmr_q(q[:15]), limit=3)
    assert str(mmr.value) == str(single.value)
    from qdrant_client.http import models as http_models

    for name in ("Mmr", "NearestQuery", "QueryRequest"):
        assert getattr(http_models, name) is getattr(models, name)


def test_query_batch_points_equals_the_loop_with_one_call_per_group(client):
    from qdrant_client import models

    col, stored = _fill(client)
    rng = np.random.default_rng(8)
    flts = [None, _cls(0), _cls(1), _cls(0), None, _cls(2)]
    reqs = []
    for i in range(30):
        v = (stored[rng.integers(0, 300)] + 0.1 * rng.standard_normal(16)).tolist()
        kind = i % 6
        if kind == 0:
            query = v
        elif kind == 1:
            query = models.NearestQuery(nearest=v)
        elif kind in (2, 3):
            query = _mmr_q(v, (0.2, 0.5, 0.8)[i % 3], (None, 40)[i % 2])
        elif kind == 4:
            query = models.RecommendQuery(recommend=models.RecommendInput(positive=[int(rng.integers(0, 300))],
                                                                          negative=[v], strategy="best_score"))
        else:
            query = (models.DiscoverQuery(discover=models.DiscoverInput(target=v, context=[(1, 2)])) if i % 4
                     else models.ContextQuery(context=[(3, 4)]))
        reqs.append(models.QueryRequest(query=query, filter=flts[i % len(flts)], limit=(4, 6)[i % 2], offset=i % 3,
                                        with_payload=i % 4 != 0, with_vector=i % 7 == 0,
                                        score_threshold=-0.5 if i % 5 == 0 else None))
    g = col._ensure_gallery()
    g.calls.clear()
    got = client.query_batch_points("m", reqs)
    calls = list(g.calls)
    want = [client.query_points("m", query=r.query, query_filter=r.filter, limit=r.limit, offset=r.offset,
                                with_payload=r.with_payload, with_vectors=r.with_vector,
                                score_threshold=r.score_threshold) for r in reqs]
    assert got == want and all(len(p.points) > 0 for p in got)
    mmr_groups = {(r.limit + r.offset, r.query.mmr.candidates_limit or r.limit + r.offset)
                  for r in reqs if isinstance(r.query, models.NearestQuery) and r.query.mmr is not None}
    mmr_calls = [c for c in calls if c[0] == "search_mmr"]
    assert len(mmr_calls) == len(mmr_groups) and {(c[2], c[3]) for c in mmr_calls} == mmr_groups
    search_ks = {r.limit + r.offset for r in reqs if not hasattr(r.query, "mmr") or r.query.mmr is None
                 if isinstance(r.query, (list, models.NearestQuery))}
    assert len([c for c in calls if c[0] == "search"]) == len(search_ks)
    assert any(c[0] == "recommend" for c in calls) and any(c[0] == "discover" for c in calls)
