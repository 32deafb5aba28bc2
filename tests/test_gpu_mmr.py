"""rbod_search_mmr (the search's kernels, then kernel K8 mmr_select) against the fp64 oracle (oracle/oracle_mmr.py):
ids identical to the oracle's on seeded data, every answer replayed step by step by ``mmr_agrees``, diversity 0 bit for
bit equal to the search's own first ``limit`` rows, and sampled queries bit for bit equal to the query sent alone."""
import numpy as np
import pytest

from oracle import oracle_mmr as OM
from oracle import oracle_np as O
from oracle import oracle_reco as OR

pytestmark = pytest.mark.gpu

DIVERSITY = np.array([0.0, 0.3, 0.5, 1.0])


@pytest.fixture(scope="module")
def G():
    from retrieval_based_object_detection_b200 import Gallery

    return Gallery


def _gallery(G, metric, dtype, n, dim, seed, copies=1):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n // copies, dim)).astype(np.float32)
    if copies > 1:   # sources x noisy copies, like augmented crops
        x = np.repeat(x, copies, axis=0) + 0.1 * rng.standard_normal((n // copies * copies, dim)).astype(np.float32)
    if metric != "cosine":
        x *= rng.uniform(0.5, 1.5, (len(x), 1)).astype(np.float32)
    g = G(dim, dtype=dtype, metric=metric, capacity=len(x))
    g.upsert(x)
    return g, g.get_rows(np.arange(len(x)))


def _queries(stored, Q, seed):
    rng = np.random.default_rng(seed)
    q = stored[rng.integers(0, len(stored), Q)].astype(np.float64)
    q += 0.3 * np.abs(stored).mean() * rng.standard_normal(q.shape)
    return q.astype(np.float32)


def _check(g, stored, metric, q, limit, L, div, masks=None, ids=None, thr=None, exact_ids=True, prepared=None,
           qkeys=None):
    if qkeys is None:
        qkeys = OR.example_keys(q, stored, metric)   # one pass over the gallery for every query
    words = None if masks is None else np.stack([O.pack_row_mask(m) for m in masks])
    res = g.search_mmr(q, limit, L, div, score_threshold=thr, row_mask=words, mask_of_query=ids, want_keys=True)
    pad = np.inf if metric in ("euclid", "manhattan") else -np.inf
    for i in range(len(q)):
        allowed = None if ids is None or ids[i] < 0 else masks[ids[i]]
        t = None if thr is None else float(np.broadcast_to(thr, (len(q),))[i])
        d = float(np.broadcast_to(div, (len(q),))[i])
        prep = prepared[i] if prepared is not None else OM.prepare(q[i], stored, L, metric, allowed, t, qkeys[i])
        assert OM.mmr_agrees(res.rows[i], q[i], stored, limit, L, d, metric, allowed, t, prep), (i, limit, L, d)
        if exact_ids:
            want, _ = OM.mmr_select(q[i], stored, limit, L, d, metric, prepared=prep)
            assert np.array_equal(res.rows[i], want), (i, limit, L, d, res.rows[i], want)
        none = res.rows[i] < 0
        assert np.all(res.scores[i][none] == pad) and np.all(np.isneginf(res.scores64[i][none]))
        assert np.array_equal(res.scores[i][~none], OM.user_scores(res.scores64[i][~none], metric))
    return res


@pytest.mark.parametrize("metric", ["cosine", "dot", "euclid", "manhattan"])
@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32"])
def test_mmr_matches_the_oracle(G, metric, dtype):
    """20 000 rows (augmented: 20 noisy copies of each source), dims 100 / 256 / 768, limit 1 / 10 / 64, L = limit, 100,
    128 (the tensor-core pass), 200 and 1024 (the fp64 sweep), four queries with diversity 0, 0.3, 0.5 and 1."""
    dim = {"bf16": 100, "f16": 256, "f32": 768}[dtype] if metric in ("cosine", "dot") else {"bf16": 768, "f16": 100,
                                                                                             "f32": 256}[dtype]
    g, stored = _gallery(G, metric, dtype, 20_000, dim, seed=1, copies=20)
    q = _queries(stored, 4, seed=2)
    qkeys = OR.example_keys(q, stored, metric)
    for L in (100, 128, 200, 1024):
        # the oracle's 1024 x 1024 distance keys at 768 columns cost seconds a query: one query there
        sel = [3] if L == 1024 and dim == 768 and metric in ("euclid", "manhattan") else [0, 1, 2, 3]
        prepared = [OM.prepare(q[i], stored, L, metric, qkeys=qkeys[i]) for i in sel]
        for limit in (1, 10, 64):
            _check(g, stored, metric, q[sel], limit, L, DIVERSITY[sel], prepared=prepared)
    for limit in (1, 10, 64):
        _check(g, stored, metric, q, limit, limit, DIVERSITY, qkeys=qkeys)
    g.close()


@pytest.mark.parametrize("metric,dtype", [("cosine", "bf16"), ("euclid", "f32"), ("manhattan", "f16"), ("dot", "f32")])
def test_diversity_0_is_the_search_bit_for_bit(G, metric, dtype):
    g, stored = _gallery(G, metric, dtype, 20_000, 256, seed=3, copies=10)
    q = _queries(stored, 16, seed=4)
    for limit, L in ((10, 10), (10, 100), (64, 128), (10, 200), (100, 1024)):
        res = g.search_mmr(q, limit, L, 0.0, want_keys=True)
        ref = g.search(q, L, want_scores64=True)
        assert np.array_equal(res.rows, ref.rows[:, :limit])
        assert np.array_equal(res.scores.view(np.uint32), ref.scores[:, :limit].view(np.uint32))
        assert np.array_equal(res.scores64.view(np.uint64), ref.scores64[:, :limit].view(np.uint64))
    g.close()


def test_exact_duplicate_clusters(G):
    """Every stored row is there 8 times: plain search returns clusters of identical rows, MMR one row per cluster
    (identical rows tie exactly and are then penalised by their own copy)."""
    rng = np.random.default_rng(5)
    src = rng.standard_normal((2_000, 64)).astype(np.float32)
    for metric in ("cosine", "euclid"):
        g = G(64, dtype="bf16", metric=metric, capacity=16_000)
        g.upsert(np.repeat(src, 8, axis=0))
        stored = g.get_rows(np.arange(16_000))
        q = _queries(stored, 4, seed=6)
        res = _check(g, stored, metric, q, 10, 200, np.array([0.0, 0.5, 0.5, 1.0]))
        assert len(set(res.rows[0] // 8)) <= 2
        for i in (1, 2):
            assert len(set(res.rows[i] // 8)) == 10
        g.close()


def test_masks_thresholds_and_short_answers(G):
    g, stored = _gallery(G, "cosine", "f16", 20_000, 96, seed=7, copies=5)
    n = len(stored)
    rng = np.random.default_rng(8)
    masks = np.zeros((3, n), dtype=bool)
    masks[0, rng.choice(n, 6, replace=False)] = True     # fewer rows than the limit
    masks[1] = rng.random(n) < 0.05
    masks[2] = True
    q = _queries(stored, 8, seed=9)
    ids = np.array([0, -1, 1, 2, -1, 0, 1, -1], np.int32)
    div = np.resize(DIVERSITY, 8)
    qkeys = OR.example_keys(q, stored, "cosine")
    res = _check(g, stored, "cosine", q, 10, 100, div, masks, ids, qkeys=qkeys)
    assert np.all(res.rows[0][6:] == -1) and np.all(res.rows[0][:6] >= 0)
    # a threshold restricts the candidates: NaN = none
    plain = g.search(q, 100)
    thr = np.where(np.arange(8) % 2 == 0, plain.scores[:, 30], np.nan).astype(np.float32)
    res = _check(g, stored, "cosine", q, 10, 100, div, thr=thr, qkeys=qkeys)
    for i in range(0, 8, 2):
        assert np.all(res.scores[i][res.rows[i] >= 0] >= thr[i])
    thr = plain.scores[:, 4].astype(np.float32)
    res = _check(g, stored, "cosine", q, 10, 100, 0.5, thr=thr, qkeys=qkeys)
    assert np.all(res.rows[:, 5:] == -1)
    g.close()


@pytest.mark.parametrize("dim,dtype,metric", [(257, "bf16", "cosine"), (1024, "f32", "euclid"), (2304, "f16", "dot"),
                                              (4100, "f32", "cosine"), (4100, "bf16", "manhattan")])
def test_wide_and_odd_rows(G, dim, dtype, metric):
    """257 (no vector path), 1024, 2304 (the fp64 sweep answers every search) and 4100 (the picks are widened into global
    scratch instead of shared memory)."""
    g, stored = _gallery(G, metric, dtype, 3_000, dim, seed=10, copies=6)
    q = _queries(stored, 4, seed=11)
    qkeys = OR.example_keys(q, stored, metric)
    for limit, L in ((10, 100), (16, 300)):
        _check(g, stored, metric, q, limit, L, DIVERSITY, qkeys=qkeys)
    g.close()


def test_device_buffers_empty_requests_and_alone(G):
    import torch

    g = G(64, dtype="bf16", metric="euclid", capacity=16)
    res = g.search_mmr(np.zeros((0, 64), np.float32), 5, 20, 0.5)
    assert res.rows.shape == (0, 5)
    res = g.search_mmr(np.ones((3, 64), np.float32), 5, 20, 0.5, want_keys=True)
    assert np.all(res.rows == -1) and np.all(res.scores == np.inf) and np.all(np.isneginf(res.scores64))
    g.close()
    g, stored = _gallery(G, "dot", "f32", 20_000, 128, seed=12, copies=4)
    q = _queries(stored, 64, seed=13)
    masks = np.stack([np.random.default_rng(14).random(len(stored)) < 0.3, np.ones(len(stored), bool)])
    words = np.stack([O.pack_row_mask(m) for m in masks])
    ids = (np.arange(64) % 3 - 1).astype(np.int32)
    div = np.resize(DIVERSITY, 64)
    host = g.search_mmr(q, 10, 150, div, row_mask=words, mask_of_query=ids, want_keys=True)
    dev = g.search_mmr(torch.from_numpy(q).cuda(), 10, 150, div, row_mask=torch.from_numpy(words.view(np.int32)).cuda(),
                       mask_of_query=torch.from_numpy(ids).cuda(), want_keys=True)
    assert dev.rows.is_cuda
    assert np.array_equal(dev.rows.cpu().numpy(), host.rows)
    assert np.array_equal(dev.scores64.cpu().numpy().view(np.uint64), host.scores64.view(np.uint64))
    for i in (0, 1, 2, 17, 40, 63):
        one = g.search_mmr(q[i:i + 1], 10, 150, div[i], row_mask=None if ids[i] < 0 else words[ids[i]], want_keys=True)
        assert np.array_equal(one.rows[0], host.rows[i])
        assert np.array_equal(one.scores[0].view(np.uint32), host.scores[i].view(np.uint32))
        assert np.array_equal(one.scores64[0].view(np.uint64), host.scores64[i].view(np.uint64))
    g.close()


def test_client_mmr_on_a_real_gallery(tmp_path, monkeypatch):
    monkeypatch.setenv("RBOD_STORE_DIR", str(tmp_path))
    from qdrant_client import QdrantClient, models

    c = QdrantClient(location=":memory:")
    n, dim = 9_000, 48
    c.recreate_collection("m", vectors_config=models.VectorParams(size=dim, distance=models.Distance.COSINE))
    rng = np.random.default_rng(15)
    src = rng.standard_normal((n // 18, dim)).astype(np.float32)
    vecs = np.repeat(src, 18, axis=0) + 0.05 * rng.standard_normal((n, dim)).astype(np.float32)
    c.upsert("m", points=models.Batch(ids=list(range(n)), vectors=vecs.tolist(),
                                      payloads=[{"class_name": f"c{i % 5}"} for i in range(n)]))
    stored = c._root.get("m").stored_vectors(range(n))
    flt = models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value="c2"))])
    q = (src[3] + 0.2 * rng.standard_normal(dim)).astype(np.float32)
    got = c.query_points("m", query=models.NearestQuery(nearest=q.tolist(), mmr=models.Mmr(diversity=0.6,
                                                                                           candidates_limit=200)),
                         query_filter=flt, limit=10).points
    allowed = np.array([i % 5 == 2 for i in range(n)])
    rows, keys = OM.mmr_select(q, stored, 10, 200, 0.6, "cosine", allowed)
    assert [p.id for p in got] == rows.tolist()
    assert [p.score for p in got] == keys.astype(np.float32).tolist()
    plain = c.search("m", q, query_filter=flt, limit=10)
    assert len({p.id // 18 for p in got}) > len({p.id // 18 for p in plain})
    reqs = [models.QueryRequest(query=models.NearestQuery(nearest=vecs[int(a)].tolist(),
                                                          mmr=models.Mmr(diversity=(0.3, 0.7)[j % 2],
                                                                         candidates_limit=(None, 50)[j % 2])),
                                filter=flt if j % 3 == 0 else None, limit=5, offset=j % 2, with_payload=True)
            for j, a in enumerate(rng.integers(0, n, 12))]
    batch = c.query_batch_points("m", reqs)
    loop = [c.query_points("m", query=r.query, query_filter=r.filter, limit=r.limit, offset=r.offset) for r in reqs]
    assert batch == loop and all(len(p.points) == 5 for p in batch)
    c.close()
