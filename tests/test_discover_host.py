"""Discovery and context search on the host: the oracle's scoring rule on hand-built 2-D cases whose answers are known
by construction, and the client (``discover`` / ``discover_batch`` / ``query_points(query=DiscoverQuery | ContextQuery)``)
over a gallery test double that answers ``discover`` with the fp64 oracle (the device side is in
tests/test_gpu_discover.py)."""
from types import SimpleNamespace

import numpy as np
import pytest

from fakes import fake_gallery
from oracle import oracle_np as O
from oracle import oracle_discover as OD
from oracle import oracle_reco as OR


# ---------------------------------------------------------------------------------------------- the scoring rule
def _scores(examples, roles, stored, metric="dot"):
    ex = np.asarray(examples, np.float32)
    return OD.discover_score(OR.example_keys(ex, np.asarray(stored, np.float32), metric), roles, [0, len(roles)],
                             metric)[0]


def test_rows_on_the_positive_side_of_every_pair_score_exactly_zero():
    # pairs (+x, -x) and (+y, -y) under DOT: the positive quadrant satisfies both, every other row loses something
    stored = [[1, 1], [2, 0.5], [0.5, 3], [-1, 1], [1, -1], [-2, -2]]
    sc = _scores([[1, 0], [-1, 0], [0, 1], [0, -1]], [1, -1, 1, -1], stored)
    assert np.array_equal(sc[:3], [0.0, 0.0, 0.0])
    assert np.all(sc[3:] < 0)
    # one pair violated by 2 (P - N = -2 - MARGIN) scores f(-2 - MARGIN); both violated by 4 each sums the two losses
    m = OD.MARGIN
    assert sc[3] == (-2 - m) / (3 + m) and sc[4] == sc[3]
    assert sc[5] == (-4 - m) / (5 + m) + (-4 - m) / (5 + m)


def test_discovery_scores_are_an_integer_rank_plus_a_value_in_0_1():
    rng = np.random.default_rng(0)
    stored = rng.standard_normal((200, 2))
    ex = rng.standard_normal((5, 2))
    sc = _scores(ex, [0, 1, -1, 1, -1], stored, "cosine")
    rank = np.floor(sc)
    assert set(rank.tolist()) <= {-2.0, 0.0, 2.0} and len(set(rank.tolist())) == 3
    assert np.all((sc - rank > 0) & (sc - rank < 1))
    # the fractional part is s(sim(key of the target)): the order of plain search within one rank
    keys = OR.example_keys(ex[:1], stored, "cosine")[0]
    assert np.allclose(sc - rank, 0.5 * (keys / (1 + np.abs(keys)) + 1), rtol=1e-15, atol=0)


def test_a_pair_tie_counts_minus_one():
    # rows equidistant from p and n: P == N exactly, so the pair ranks -1, and the context loss is f(-MARGIN) < 0
    stored = [[0.0, 5.0], [0.0, -3.0]]
    ex = [[1, 1], [1, 0], [-1, 0]]
    for metric in ("dot", "euclid", "manhattan"):
        sc = _scores(ex, [0, 1, -1], stored, metric)
        assert np.all(np.floor(sc) == -1)
        ctx = _scores(ex[1:], [1, -1], stored, metric)
        m = OD.MARGIN
        assert np.all(ctx == -m / (1 + m))


def test_the_margin_decides_an_exact_boundary():
    # DOT with p = (1, 0), n = (0, 0): P - N = g_x, so a row at g_x = MARGIN sits exactly on the boundary (loss f(0) =
    # 0), a row at g_x = MARGIN / 2 is inside the pair's zone without the margin but loses with it
    m = OD.MARGIN
    stored = np.array([[m, 0], [m / 2, 0], [2 * m, 0], [0, 0]], np.float32)
    sc = _scores([[1, 0], [0, 0]], [1, -1], stored)
    assert sc[0] == 0.0 and sc[2] == 0.0
    assert sc[1] == (-m / 2) / (1 + m / 2) and sc[1] < 0
    assert sc[3] == -m / (1 + m)


# ---------------------------------------------------------------------------------------------- the client
class DiscFakeGallery(fake_gallery.FakeGallery):
    def discover(self, examples, roles, offsets, k, row_mask=None, mask_of_request=None, want_keys=False):
        ex = np.asarray(examples, dtype=np.float32).reshape(-1, self.dim)
        roles, offsets = np.asarray(roles, dtype=np.int8), np.asarray(offsets, dtype=np.int64)
        R, n = len(offsets) - 1, len(self._rows)
        assert len(roles) == len(ex) == offsets[-1] and offsets[0] == 0 and np.all(np.diff(offsets) >= 1)
        assert np.all(np.diff(offsets) <= 32) and set(roles.tolist()) <= {0, 1, -1} and 1 <= k <= 1024
        for r in range(R):
            rl = roles[offsets[r]:offsets[r + 1]].tolist()
            body = rl[1:] if rl[0] == 0 else rl
            assert body == [1, -1] * (len(body) // 2)
        if row_mask is None:
            allowed, n_masks = None, 0
        else:
            masks = np.asarray(row_mask, dtype=np.uint32).reshape(-1, (n + 31) // 32)
            ids = np.zeros(R, dtype=np.int32) if mask_of_request is None else np.asarray(mask_of_request)
            allowed = [None if i < 0 else O.unpack_row_mask(masks[i], n) for i in ids]
            n_masks = len(masks)
        self.calls.append(("discover", R, k, n_masks))
        s, i = OD.discover_topk(ex, roles, offsets, self._rows, k, self.metric, allowed)
        return SimpleNamespace(scores=s.astype(np.float32), rows=i, scores64=s if want_keys else None, stats={})


@pytest.fixture()
def client(store_dir, monkeypatch):
    import retrieval_based_object_detection_b200 as pkg
    import retrieval_based_object_detection_b200.gallery as gallery

    monkeypatch.setattr(gallery, "Gallery", DiscFakeGallery)
    monkeypatch.setattr(pkg, "Gallery", DiscFakeGallery)
    from qdrant_client import QdrantClient

    return QdrantClient(host="localhost", port=6333)


def _fill(client, distance="COSINE", n=300, dim=16):
    from qdrant_client import models

    client.recreate_collection("d", vectors_config=models.VectorParams(size=dim, distance=getattr(models.Distance, distance)))
    rng = np.random.default_rng(5)
    vecs = rng.standard_normal((n, dim)).astype(np.float32)
    client.upsert("d", points=models.Batch(ids=list(range(n)), vectors=vecs.tolist(),
                                           payloads=[{"class_name": f"c{i % 7}"} for i in range(n)]))
    col = client._root.get("d")
    return col, col.stored_vectors(range(n))


def _cls(j):
    from qdrant_client import models

    return models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value=f"c{j}"))])


def _pair(p, n):
    from qdrant_client import models

    return models.ContextExamplePair(positive=p, negative=n)


@pytest.mark.parametrize("distance", ["COSINE", "EUCLID"])
def test_ids_and_vectors_match_the_oracle(client, distance):
    col, stored = _fill(client, distance)
    metric = distance.lower()
    raw = np.random.default_rng(6).standard_normal((2, 16)).astype(np.float32)
    got = client.discover("d", target=raw[0].tolist(), context=[_pair(3, 17), _pair(raw[1].tolist(), 40)], limit=12)
    ex = np.stack([raw[0], stored[3], stored[17], raw[1], stored[40]])
    s, i = OD.discover_topk(ex, [0, 1, -1, 1, -1], [0, 5], stored, 15, metric)
    keep = ~np.isin(i[0], [3, 17, 40])
    assert [p.id for p in got] == i[0][keep][:12].tolist()
    assert [p.score for p in got] == s[0][keep][:12].astype(np.float32).tolist()
    assert all(p.payload == {"class_name": f"c{p.id % 7}"} for p in got)
    # a context search: scores <= 0, ties at 0 ordered by point
    got = client.discover("d", context=[_pair(5, 6), _pair(7, raw[1].tolist())], limit=20)
    s, i = OD.discover_topk(np.stack([stored[5], stored[6], stored[7], raw[1]]), [1, -1, 1, -1], [0, 4], stored,
                            23, metric)
    keep = ~np.isin(i[0], [5, 6, 7])
    assert [p.id for p in got] == i[0][keep][:20].tolist()
    assert all(p.score <= 0 for p in got)


def test_example_ids_never_appear_even_inside_the_top_k(client):
    col, stored = _fill(client)
    g = col._ensure_gallery()
    # target 10 is the best hit of its own discovery (s(1) over rank 0); the positive 11 ranks high as well
    raw = g.discover(stored[[10, 11, 12]], [0, 1, -1], [0, 3], 5)
    assert 10 in set(np.asarray(raw.rows[0]).tolist())
    got = client.discover("d", target=10, context=[(11, 12)], limit=5)
    assert len(got) == 5 and not {10, 11, 12} & {p.id for p in got}
    # an id given twice is fetched once
    g.calls.clear()
    client.discover("d", target=10, context=[(11, 12), (10, 12)], limit=5)
    assert [c[2] for c in g.calls if c[0] == "discover"] == [8]


def test_unknown_id_names_it(client):
    _fill(client)
    with pytest.raises(ValueError, match="discover: point 999 not found in collection 'd'"):
        client.discover("d", target=999, context=[(1, 2)])
    with pytest.raises(ValueError, match="12345678-1234-5678-1234-567812345678"):
        client.discover("d", context=[(1, "12345678-1234-5678-1234-567812345678")])


@pytest.mark.parametrize("distance", ["COSINE", "MANHATTAN"])
def test_offset_and_score_threshold(client, distance):
    from qdrant_client import models

    _fill(client, distance)
    for target in (1, None):
        full = client.discover("d", target=target, context=[(2, 3), (4, 5)], limit=40)
        assert client.discover("d", target=target, context=[(2, 3), (4, 5)], limit=5, offset=3) == full[3:8]
        thr = full[9].score
        q = (models.DiscoverQuery(discover=models.DiscoverInput(target=target, context=[(2, 3), (4, 5)]))
             if target is not None else models.ContextQuery(context=[(2, 3), (4, 5)]))
        got = client.query_points("d", query=q, limit=40, score_threshold=thr).points
        # larger-is-better for every distance: the threshold keeps scores >= it
        assert got == [p for p in full if p.score >= thr] and len(got) >= 10


def test_discover_batch_equals_the_loop_with_one_call_per_fetch_and_one_mask_per_filter(client):
    from qdrant_client import models

    col, _ = _fill(client)
    rng = np.random.default_rng(8)
    flts = [None, _cls(0), _cls(1), _cls(0), None, _cls(2)]
    reqs = []
    for i in range(24):
        ids = [int(x) for x in rng.choice(300, 5, replace=False)]
        target = (ids[0] if i % 4 else rng.standard_normal(16).tolist()) if i % 3 else None
        pairs = [models.ContextExamplePair(positive=ids[1], negative=ids[2])]
        if i % 2:
            pairs.append(models.ContextExamplePair(positive=ids[3], negative=ids[4]))
        reqs.append(models.DiscoverRequest(target=target, context=pairs, filter=flts[i % len(flts)],
                                           limit=(3, 6)[i % 2], offset=i % 3, with_payload=i % 4 != 0,
                                           with_vector=i % 7 == 0))
    g = col._ensure_gallery()
    g.calls.clear()
    got = client.discover_batch("d", reqs)
    calls = [c for c in g.calls if c[0] == "discover"]
    want = [client.discover("d", r.target, r.context, r.filter, None, r.limit, r.offset, bool(r.with_payload),
                            bool(r.with_vector)) for r in reqs]
    assert got == want and all(len(p) > 0 for p in got)
    fetch = {}
    for r in reqs:
        n_ids = len({x for p in r.context for x in (p.positive, p.negative)} |
                    ({r.target} if isinstance(r.target, int) else set()))
        fetch.setdefault(r.limit + r.offset + n_ids, []).append(r)
    assert len(calls) == len(fetch)
    for c in calls:
        members = fetch[c[2]]
        assert c[1] == len(members)
        assert c[3] == len({repr(r.filter) for r in members if r.filter is not None})


def test_query_forms_single_pairs_and_tuples(client):
    from qdrant_client import models
    from qdrant_client.http import models as http_models

    _fill(client)
    for name in ("ContextExamplePair", "DiscoverRequest", "ContextPair", "DiscoverInput", "DiscoverQuery",
                 "ContextQuery"):
        assert getattr(http_models, name) is getattr(models, name)
    want = client.discover("d", target=1, context=[_pair(2, 3)], query_filter=_cls(1), limit=4, offset=1)
    assert len(want) == 4 and all(p.payload["class_name"] == "c1" for p in want)
    q = models.DiscoverQuery(discover=models.DiscoverInput(target=1, context=[models.ContextPair(positive=2, negative=3)]))
    assert client.query_points("d", query=q, query_filter=_cls(1), limit=4, offset=1).points == want
    q = models.DiscoverQuery(discover=models.DiscoverInput(target=1, context=models.ContextPair(positive=2, negative=3)))
    assert client.query_points("d", query=q, query_filter=_cls(1), limit=4, offset=1).points == want
    # a single pair, a list of one pair, a 2-tuple, a list of 2-tuples
    for ctx in (_pair(2, 3), [_pair(2, 3)], (2, 3), [(2, 3)], [models.ContextPair(positive=2, negative=3)]):
        assert client.discover("d", target=1, context=ctx, query_filter=_cls(1), limit=4, offset=1) == want
    two = client.discover("d", context=[(2, 3), (4, 5)], limit=6)
    assert client.discover("d", context=((2, 3), (4, 5)), limit=6) == two
    assert client.query_points("d", query=models.ContextQuery(context=[models.ContextPair(positive=2, negative=3),
                                                                       (4, 5)]), limit=6).points == two


def test_limits_and_unsupported_arguments(client):
    _fill(client)
    client.discover("d", context=[(i, i + 100) for i in range(16)])
    client.discover("d", target=0, context=[(i, i + 100) for i in range(1, 16)])
    with pytest.raises(ValueError, match="at most 32 examples .*got 33"):
        client.discover("d", target=0, context=[(i, i + 100) for i in range(1, 17)])
    client.discover("d", target=1, context=[(2, 3)], limit=1020, offset=1)
    with pytest.raises(ValueError, match="1025 exceeds 1024"):
        client.discover("d", target=1, context=[(2, 3)], limit=1020, offset=2)
    with pytest.raises(ValueError, match="needs a target or at least one context pair"):
        client.discover("d")
    with pytest.raises(ValueError, match="needs a target or at least one context pair"):
        client.discover("d", context=[])
    with pytest.raises(ValueError, match="context pair is"):
        client.discover("d", context=[(1, 2, 3)])
    with pytest.raises(ValueError, match="named vectors"):
        client.discover("d", target=1, using="image")
    with pytest.raises(ValueError, match="lookup_from"):
        client.discover("d", target=1, lookup_from={"collection": "other"})
    from qdrant_client import models

    with pytest.raises(ValueError, match="named vectors"):
        client.query_points("d", query=models.ContextQuery(context=(1, 2)), using="image")
    with pytest.raises(ValueError) as single:
        client.search("d", [0.1] * 15, limit=3)
    with pytest.raises(ValueError) as disc:
        client.discover("d", target=[0.1] * 15)
    assert str(disc.value) == str(single.value)
    assert client.discover("d", target=1, limit=0) == []
