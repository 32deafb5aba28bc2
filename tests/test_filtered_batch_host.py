"""Host side of batched filtered search: ``search_batch(requests=...)`` and ``query_filters`` compile each distinct
filter once and make one gallery search per distinct ``limit + offset``, with one mask per query.  The gallery is a
test double that answers every query with the oracle and its own mask (the device side is in
tests/test_gpu_masked_search.py)."""
import numpy as np
import pytest

from fakes import fake_gallery
from oracle import oracle_np as O


class MaskedFakeGallery(fake_gallery.FakeGallery):
    def search(self, queries, k, row_mask=None, want_scores64=False, out=None, stream=None, mask_of_query=None):
        if mask_of_query is None:
            return super().search(queries, k, row_mask, want_scores64, out, stream)
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        ids = np.asarray(mask_of_query, dtype=np.int32)
        masks = np.asarray(row_mask, dtype=np.uint32).reshape(-1, (len(self._rows) + 31) // 32)
        assert ids.shape == (len(q),) and ids.min() >= -1 and ids.max() < len(masks)
        self.calls.append(("search_masks", len(q), k, len(masks)))
        scores = np.empty((len(q), k), dtype=np.float32)
        rows = np.empty((len(q), k), dtype=np.int64)
        for i in range(len(q)):
            one = fake_gallery.FakeGallery.search(self, q[i:i + 1], k, None if ids[i] < 0 else masks[ids[i]])
            self.calls.pop()
            scores[i], rows[i] = one.scores[0], one.rows[0]
        return type(one)(scores=scores, rows=rows, scores64=scores.astype(np.float64), stats={})


@pytest.fixture()
def client(store_dir, monkeypatch):
    import retrieval_based_object_detection_b200 as pkg
    import retrieval_based_object_detection_b200.gallery as gallery

    monkeypatch.setattr(gallery, "Gallery", MaskedFakeGallery)
    monkeypatch.setattr(pkg, "Gallery", MaskedFakeGallery)
    from qdrant_client import QdrantClient

    return QdrantClient(host="localhost", port=6333)


def _fill(client, n=300, dim=16):
    from qdrant_client import models

    client.recreate_collection("b", vectors_config=models.VectorParams(size=dim, distance=models.Distance.COSINE))
    rng = np.random.default_rng(2)
    vecs = rng.standard_normal((n, dim)).astype(np.float32)
    client.upsert("b", points=models.Batch(ids=list(range(n)), vectors=vecs.tolist(),
                                           payloads=[{"class_name": f"c{i % 7}", "seg": i % 3 == 0} for i in range(n)]))
    return vecs


def _filters():
    from qdrant_client import models

    def cls(j):
        return models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value=f"c{j}"))])

    return [None, cls(0), cls(1), cls(2),
            models.Filter(must_not=[models.FieldCondition(key="seg", match=models.MatchValue(value=True))]),
            cls(0),                                                   # equal to an earlier filter
            models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value="none"))])]


def _gallery(client):
    return client._root.get("b")._ensure_gallery()


def test_requests_equal_the_per_request_loop(client):
    from qdrant_client import models

    _fill(client)
    rng = np.random.default_rng(3)
    flts = _filters()
    reqs = [models.SearchRequest(vector=rng.standard_normal(16).tolist(), filter=flts[i % len(flts)],
                                 limit=(3, 5, 400)[i % 3], offset=(0, 2)[i % 2], with_payload=i % 4 != 0,
                                 with_vector=i % 5 == 0, score_threshold=0.1 if i % 6 == 0 else None)
            for i in range(40)]
    reqs.append(models.SearchRequest(vector=rng.standard_normal(16).tolist(), limit=0))
    got = client.search_batch("b", requests=reqs)
    want = [client.search("b", r.vector, r.filter, r.limit, r.offset or 0, bool(r.with_payload), bool(r.with_vector),
                          r.score_threshold) for r in reqs]
    assert got == want
    assert got[-1] == [] and any(len(p) > 0 for p in got)


def test_one_gallery_search_per_limit_plus_offset_and_one_mask_per_filter(client):
    from qdrant_client import models

    _fill(client)
    rng = np.random.default_rng(4)
    flts = _filters()
    # limit + offset: 5, 5, 5, 10 -> two groups; the 7 filters hold 5 distinct ones (cls(0) twice, one None)
    shapes = [(5, 0), (3, 2), (4, 1), (10, 0)]
    reqs = [models.SearchRequest(vector=rng.standard_normal(16).tolist(), filter=flts[i % len(flts)],
                                 limit=shapes[i % 4][0], offset=shapes[i % 4][1]) for i in range(28)]
    g = _gallery(client)
    g.calls.clear()
    client.search_batch("b", requests=reqs)
    searches = [c for c in g.calls if c[0].startswith("search")]
    assert sorted(c[1:3] for c in searches) == [(7, 10), (21, 5)]
    assert {c[0] for c in searches} == {"search_masks"}
    assert [c[3] for c in searches] == [5, 5]                     # both groups see every filter: 5 distinct masks
    # all filters None: the plain search
    g.calls.clear()
    client.search_batch("b", requests=[models.SearchRequest(vector=rng.standard_normal(16).tolist(), limit=4)] * 3)
    assert [c[0] for c in g.calls] == ["search"]


def test_query_filters_tensor_form(client):
    vecs = _fill(client)
    flts = _filters()
    q = vecs[:len(flts)] + 0.01
    scores, ids = client.search_batch("b", queries=q, k=4, query_filters=flts)
    for i, f in enumerate(flts):
        s1, i1 = client.search_batch("b", queries=q[i:i + 1], k=4, row_filter=f)
        assert ids[i] == i1[0] and np.array_equal(scores[i], s1[0])
    col = client._root.get("b")
    allowed = O.unpack_row_mask(col.filter_mask(flts[1]), len(col.ids))
    assert all(allowed[col.slot_of[pid]] for pid in ids[1] if pid is not None)
    with pytest.raises(ValueError):
        client.search_batch("b", queries=q, k=4, row_filter=flts[1], query_filters=flts)
    with pytest.raises(ValueError):
        client.search_batch("b", queries=q, k=4, query_filters=flts[:2])


def test_wrong_dimension_raises_the_same_error(client):
    from qdrant_client import models

    _fill(client)
    good = models.SearchRequest(vector=[0.1] * 16, limit=3)
    bad = models.SearchRequest(vector=[0.1] * 15, limit=3)
    with pytest.raises(ValueError) as single:
        client.search("b", bad.vector, limit=3)
    with pytest.raises(ValueError) as batch:
        client.search_batch("b", requests=[good, bad])
    assert str(batch.value) == str(single.value)
