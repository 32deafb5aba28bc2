"""rbod_discover (kernel K7, discovery and context search) against the fp64 oracle (oracle/oracle_discover.py
``discover_score``): scores within rtol 1e-12 and ids equal to the oracle's, except among rows the oracle scores within
that tolerance of each other (see ``agrees``); sampled requests bit for bit equal to the same request sent alone.

A context loss is f(sim(P) - sim(N) - MARGIN): near a pair's boundary it is the small difference of two keys, so two
fp64 sums taken in different orders agree on it only to a few ulps of the keys, not relative to the loss.  The
comparison therefore adds an absolute tolerance of 1e-12 times the largest |key| of the request."""
import numpy as np
import pytest

from oracle import oracle_np as O
from oracle import oracle_discover as OD
from oracle import oracle_reco as OR

pytestmark = pytest.mark.gpu

# (has a target, pairs): discovery, context and target-only requests; passes of 32 slots and of at most 8 (NS = 8)
SHAPES = [(True, 15), (False, 1), (True, 0), (True, 1), (False, 16), (False, 3), (True, 9), (False, 6), (True, 3),
          (True, 0), (False, 2), (True, 14), (False, 1), (True, 2)]


@pytest.fixture(scope="module")
def G():
    from retrieval_based_object_detection_b200 import Gallery

    return Gallery


def _gallery(G, metric, dtype, n, dim, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    if metric != "cosine":
        x *= rng.uniform(0.2, 2.0, (n, 1)).astype(np.float32)
    g = G(dim, dtype=dtype, metric=metric, capacity=n)
    g.upsert(x)
    return g, g.get_rows(np.arange(n))


def _requests(stored, shapes, seed):
    """Half the examples are stored rows, half perturbed stored rows."""
    rng = np.random.default_rng(seed)
    n, dim = stored.shape
    ex, roles, sizes = [], [], []
    for target, pairs in shapes:
        rl = ([0] if target else []) + [1, -1] * pairs
        rows = stored[rng.integers(0, n, len(rl))].copy()
        noisy = rng.random(len(rl)) < 0.5
        rows[noisy] += 0.3 * rng.standard_normal((int(noisy.sum()), dim)).astype(np.float32) * np.abs(stored).mean()
        ex.append(rows)
        roles.append(np.asarray(rl, np.int8))
        sizes.append(len(rl))
    offsets = np.zeros(len(shapes) + 1, np.int64)
    np.cumsum(sizes, out=offsets[1:])
    return np.concatenate(ex), np.concatenate(roles), offsets


def _mask_set(n, seed):
    """Masks that allow one row, five rows (fewer than k), 1 % and every row."""
    rng = np.random.default_rng(seed)
    m = np.zeros((4, n), dtype=bool)
    m[0, rng.integers(0, n)] = True
    m[1, rng.choice(n, 5, replace=False)] = True
    m[2] = rng.random(n) < 0.01
    m[3] = True
    return m


def _agrees(got_rows, got_keys, scores, want_keys, want_rows, atol):
    """``OR.agrees`` (rtol 1e-12) with an absolute tolerance ``atol`` added to every score comparison."""
    got_rows, got_keys = np.asarray(got_rows), np.asarray(got_keys, dtype=np.float64)
    valid = np.asarray(want_rows) >= 0
    if not np.array_equal(got_rows >= 0, valid) or not np.all(np.isneginf(got_keys[~valid])):
        return False
    g, gk, wk = got_rows[valid], got_keys[valid], np.asarray(want_keys)[valid]
    if len(np.unique(g)) != len(g) or np.any((gk[1:] > gk[:-1]) | ((gk[1:] == gk[:-1]) & (g[1:] < g[:-1]))):
        return False
    return bool(np.allclose(scores[g], wk, rtol=1e-12, atol=atol) and np.allclose(gk, wk, rtol=1e-12, atol=atol))


def _oracle(ex, roles, offsets, stored, metric):
    """-> (scores [R, n], absolute tolerance per request: 1e-12 x the largest |key| of its examples)."""
    keys = OR.example_keys(ex, stored, metric)
    atol = np.array([1e-12 * max(1.0, np.abs(keys[offsets[r]:offsets[r + 1]]).max()) for r in range(len(offsets) - 1)])
    return OD.discover_score(keys, roles, offsets, metric), atol


def _check(g, stored, metric, ex, roles, offsets, ks, masks=None, ids=None, alone=(0,), oracle=None):
    R = len(offsets) - 1
    words = None if masks is None else np.stack([O.pack_row_mask(m) for m in masks])
    allowed = None if masks is None else [None if i < 0 else masks[i] for i in ids]
    scores, atol = _oracle(ex, roles, offsets, stored, metric) if oracle is None else oracle
    for k in ks:
        res = g.discover(ex, roles, offsets, k, row_mask=words, mask_of_request=ids, want_keys=True)
        assert res.stats["queries"] == R and res.stats["sweep_queries"] == R
        for r in range(R):
            ws, wi = O.topk_from_scores(scores[r:r + 1], k, row_mask=None if allowed is None else allowed[r])
            assert _agrees(res.rows[r], res.scores64[r], scores[r], ws[0], wi[0], atol[r]), (k, r, res.rows[r], wi[0])
            assert np.all(np.isneginf(res.scores[r][wi[0] < 0]))
        assert np.array_equal(res.scores, res.scores64.astype(np.float32))
        for r in alone:
            a, b = offsets[r], offsets[r + 1]
            one = g.discover(ex[a:b], roles[a:b], [0, b - a], k,
                             row_mask=None if ids is None or ids[r] < 0 else words[ids[r]], want_keys=True)
            assert np.array_equal(one.rows[0], res.rows[r]), (k, r)
            assert np.array_equal(one.scores[0].view(np.uint32), res.scores[r].view(np.uint32)), (k, r)
            assert np.array_equal(one.scores64[0].view(np.uint64), res.scores64[r].view(np.uint64)), (k, r)
    return scores, atol


@pytest.mark.parametrize("metric", ["cosine", "dot", "euclid", "manhattan"])
@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32"])
def test_discover_matches_the_oracle(G, metric, dtype):
    """20 000 rows (the sample pass runs), 100 columns (a partial chunk), discovery, context and target-only requests
    packed into passes of 32 and of at most 8 slots, k = 1, 10, 100, 1024, unfiltered and with a mask per request."""
    g, stored = _gallery(G, metric, dtype, 20_000, 100, seed=1)
    ex, roles, offsets = _requests(stored, SHAPES, seed=2)
    R = len(SHAPES)
    oracle = _check(g, stored, metric, ex, roles, offsets, (1, 10, 100, 1024), alone=(1, 2, 6, 13))
    masks = _mask_set(len(stored), seed=3)
    ids = (np.arange(R) % (len(masks) + 1) - 1).astype(np.int32)
    _check(g, stored, metric, ex, roles, offsets, (10, 100), masks, ids, alone=(1, 2, 3, 4), oracle=oracle)
    g.close()


@pytest.mark.parametrize("dim,dtype", [(1024, "bf16"), (2304, "f32"), (2304, "f16")])
def test_wide_rows(G, dim, dtype):
    g, stored = _gallery(G, "cosine", dtype, 9_000, dim, seed=4)
    ex, roles, offsets = _requests(stored, [(True, 1), (False, 16), (True, 0), (False, 4)], seed=5)
    _check(g, stored, "cosine", ex, roles, offsets, (10, 200), alone=(0, 2))
    g.close()


def test_more_than_32_requests_and_many_passes(G):
    g, stored = _gallery(G, "euclid", "bf16", 12_000, 64, seed=6)
    ex, roles, offsets = _requests(stored, [(True, 0)] * 20 + [(False, 1)] * 20 + [(True, 1)] * 10 + [(False, 16)],
                                   seed=7)
    _check(g, stored, "euclid", ex, roles, offsets, (7,), alone=(0, 25, 45, 50))
    g.close()


def test_context_plateau_overflows_and_resweeps(G):
    """A context pair whose positive side holds about half of 40 000 rows: all of them score exactly 0, far more than
    the 8192 rows a list holds, so the sweep tightens to the k-th (score, row) pair and sweeps again.  The answer is the
    k lowest row slots of the plateau."""
    g, stored = _gallery(G, "dot", "f32", 40_000, 32, seed=8)
    p = np.zeros((1, 32), np.float32)
    p[0, 0] = 1.0
    ex = np.concatenate([p, -p])
    roles = np.array([1, -1], np.int8)
    zone = np.nonzero(stored[:, 0].astype(np.float64) >= OD.MARGIN / 2)[0]
    assert len(zone) > 15_000
    for k in (10, 1024):
        res = g.discover(ex, roles, [0, 2], k, want_keys=True)
        assert res.stats["fallback_queries"] > 0
        assert np.array_equal(res.rows[0], zone[:k]) and np.all(res.scores64[0] == 0.0)
    _check(g, stored, "dot", ex, roles, np.array([0, 2]), (10,), alone=())
    g.close()


def test_target_only_discovery_is_plain_search(G):
    g, stored = _gallery(G, "cosine", "f32", 20_000, 96, seed=9)
    rng = np.random.default_rng(10)
    q = (stored[rng.integers(0, len(stored), 6)] + 0.2 * rng.standard_normal((6, 96))).astype(np.float32)
    for k in (10, 100):
        res = g.discover(q, np.zeros(6, np.int8), np.arange(7), k, want_keys=True)
        ref = g.search(q, k, want_scores64=True)
        keys = OR.example_keys(q, stored, "cosine")
        for r in range(6):
            if not np.array_equal(res.rows[r], ref.rows[r]):
                # only rows whose search keys lie within 1e-12 of each other may swap
                a, b = keys[r][res.rows[r]], keys[r][ref.rows[r]]
                assert np.allclose(np.sort(a), np.sort(b), rtol=1e-12, atol=0), r
    g.close()


def test_empty_requests_empty_gallery_and_device_inputs(G):
    import torch

    g = G(64, dtype="bf16", metric="cosine", capacity=16)
    res = g.discover(np.zeros((0, 64), np.float32), np.zeros(0, np.int8), [0], 5)
    assert res.rows.shape == (0, 5)
    res = g.discover(np.ones((3, 64), np.float32), [0, 1, -1], [0, 3], 5, want_keys=True)
    assert np.all(res.rows == -1) and np.all(np.isneginf(res.scores)) and np.all(np.isneginf(res.scores64))
    g.close()
    g, stored = _gallery(G, "dot", "f16", 15_000, 200, seed=11)
    ex, roles, offsets = _requests(stored, [(True, 2), (False, 1), (False, 16), (True, 0)], seed=12)
    masks = _mask_set(len(stored), seed=13)
    words = np.stack([O.pack_row_mask(m) for m in masks])
    ids = np.array([3, -1, 2, 0], np.int32)
    host = g.discover(ex, roles, offsets, 50, row_mask=words, mask_of_request=ids, want_keys=True)
    dev = g.discover(torch.from_numpy(ex).cuda(), roles, offsets, 50, row_mask=torch.from_numpy(words.view(np.int32)).cuda(),
                     mask_of_request=torch.from_numpy(ids).cuda(), want_keys=True)
    assert dev.rows.is_cuda
    assert np.array_equal(dev.rows.cpu().numpy(), host.rows)
    assert np.array_equal(dev.scores64.cpu().numpy().view(np.uint64), host.scores64.view(np.uint64))
    _check(g, stored, "dot", ex, roles, offsets, (50,), masks, ids, alone=())
    g.close()


def test_client_discover_on_a_real_gallery(tmp_path, monkeypatch):
    monkeypatch.setenv("RBOD_STORE_DIR", str(tmp_path))
    from qdrant_client import QdrantClient, models

    c = QdrantClient(location=":memory:")
    n, dim = 10_000, 48
    c.recreate_collection("d", vectors_config=models.VectorParams(size=dim, distance=models.Distance.COSINE))
    rng = np.random.default_rng(14)
    c.upsert("d", points=models.Batch(ids=list(range(n)), vectors=rng.standard_normal((n, dim)).astype(np.float32).tolist(),
                                      payloads=[{"class_name": f"c{i % 5}"} for i in range(n)]))
    col = c._root.get("d")
    stored = col.stored_vectors(range(n))
    flt = models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value="c2"))])
    got = c.discover("d", target=10, context=[models.ContextExamplePair(positive=11, negative=12)], query_filter=flt,
                     limit=7)
    allowed = np.array([i % 5 == 2 for i in range(n)])
    allowed[[10, 11, 12]] = False
    s, i = OD.discover_topk(stored[[10, 11, 12]], [0, 1, -1], [0, 3], stored, 7, "cosine", [allowed])
    assert [p.id for p in got] == i[0].tolist()
    assert np.allclose([p.score for p in got], s[0], rtol=1e-7)
    reqs = [models.DiscoverRequest(target=int(a) if j % 3 else None,
                                   context=[(int(b), rng.standard_normal(dim).tolist())] * (1 + j % 2),
                                   filter=flt if j % 4 == 0 else None, limit=5, offset=j % 2, with_payload=True)
            for j, (a, b) in enumerate(rng.integers(0, n, (12, 2)))]
    batch = c.discover_batch("d", reqs)
    loop = [c.discover("d", r.target, r.context, r.filter, None, r.limit, r.offset) for r in reqs]
    assert batch == loop and all(len(p) == 5 for p in batch)
    c.close()
