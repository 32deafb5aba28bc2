"""rbod_recommend (kernel K6, best_score) against the fp64 oracle (oracle/oracle_reco.py): scores within rtol 1e-12 and
ids equal to the oracle's, except among rows the oracle scores within 1e-12 of each other (examples are often stored
rows, which score s(1) against themselves give or take an ulp, so their order differs between two summation orders);
sampled requests bit for bit equal to the same request sent alone."""
import numpy as np
import pytest

from oracle import oracle_np as O
from oracle import oracle_reco as OR

pytestmark = pytest.mark.gpu

# request sizes: passes of 32 slots, passes of 8 or fewer (NS = 8), and several requests per pass
SIZES = [32, 1, 2, 3, 32, 5, 20, 13, 8, 1, 1, 30, 4, 2]


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


def _requests(stored, sizes, seed):
    """Positives only, negatives only and mixed requests; half the examples are stored rows, half perturbed rows."""
    rng = np.random.default_rng(seed)
    n, dim = stored.shape
    ex, signs = [], []
    for r, m in enumerate(sizes):
        rows = stored[rng.integers(0, n, m)].copy()
        noisy = rng.random(m) < 0.5
        rows[noisy] += 0.3 * rng.standard_normal((int(noisy.sum()), dim)).astype(np.float32) * np.abs(stored).mean()
        ex.append(rows)
        kind = r % 3
        s = np.ones(m, np.int8) if kind == 0 else (-np.ones(m, np.int8) if kind == 1 else
                                                   np.where(rng.random(m) < 0.5, 1, -1).astype(np.int8))
        if kind == 2 and m > 1:
            s[0], s[-1] = 1, -1
        signs.append(s)
    offsets = np.zeros(len(sizes) + 1, np.int64)
    np.cumsum(sizes, out=offsets[1:])
    return np.concatenate(ex), np.concatenate(signs), offsets


def _mask_set(n, seed):
    """Masks that allow one row, five rows (fewer than k), 1 % and every row."""
    rng = np.random.default_rng(seed)
    m = np.zeros((4, n), dtype=bool)
    m[0, rng.integers(0, n)] = True
    m[1, rng.choice(n, 5, replace=False)] = True
    m[2] = rng.random(n) < 0.01
    m[3] = True
    return m


def _check(g, stored, metric, ex, signs, offsets, ks, masks=None, ids=None, alone=(0,), scores=None):
    R = len(offsets) - 1
    words = None if masks is None else np.stack([O.pack_row_mask(m) for m in masks])
    allowed = None if masks is None else [None if i < 0 else masks[i] for i in ids]
    if scores is None:
        scores = OR.best_score(OR.example_keys(ex, stored, metric), signs, offsets, metric)
    for k in ks:
        res = g.recommend(ex, signs, offsets, k, row_mask=words, mask_of_request=ids, want_keys=True)
        assert res.stats["queries"] == R and res.stats["sweep_queries"] == R
        for r in range(R):
            ws, wi = O.topk_from_scores(scores[r:r + 1], k, row_mask=None if allowed is None else allowed[r])
            # ids equal to the oracle's, except among rows it scores within 1e-12 of each other (see OR.agrees)
            assert OR.agrees(res.rows[r], res.scores64[r], scores[r], ws[0], wi[0]), (k, r, res.rows[r], wi[0])
            same = res.rows[r] == wi[0]
            assert np.allclose(ws[0][~same], scores[r][res.rows[r][~same]], rtol=1e-12, atol=0)
            assert np.all(np.isneginf(res.scores[r][wi[0] < 0]))
        assert np.array_equal(res.scores, res.scores64.astype(np.float32))
        for r in alone:
            a, b = offsets[r], offsets[r + 1]
            one = g.recommend(ex[a:b], signs[a:b], [0, b - a], k, row_mask=None if ids is None or ids[r] < 0 else words[ids[r]],
                              want_keys=True)
            assert np.array_equal(one.rows[0], res.rows[r]), (k, r)
            assert np.array_equal(one.scores[0].view(np.uint32), res.scores[r].view(np.uint32)), (k, r)
            assert np.array_equal(one.scores64[0].view(np.uint64), res.scores64[r].view(np.uint64)), (k, r)
    return scores


@pytest.mark.parametrize("metric", ["cosine", "dot", "euclid", "manhattan"])
@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32"])
def test_best_score_matches_the_oracle(G, metric, dtype):
    """20 000 rows (the sample pass runs), 100 columns (a partial chunk), requests of 1 to 32 examples packed into
    passes of 32 and of at most 8 slots, k = 1, 10, 100, 1024, unfiltered and with a mask per request."""
    g, stored = _gallery(G, metric, dtype, 20_000, 100, seed=1)
    ex, signs, offsets = _requests(stored, SIZES, seed=2)
    R = len(SIZES)
    scores = _check(g, stored, metric, ex, signs, offsets, (1, 10, 100, 1024), alone=(1, 6, 13))
    masks = _mask_set(len(stored), seed=3)
    ids = (np.arange(R) % (len(masks) + 1) - 1).astype(np.int32)
    _check(g, stored, metric, ex, signs, offsets, (10, 100), masks, ids, alone=(1, 2, 3, 4), scores=scores)
    g.close()


@pytest.mark.parametrize("dim,dtype", [(1024, "bf16"), (2304, "f32"), (2304, "f16")])
def test_wide_rows(G, dim, dtype):
    g, stored = _gallery(G, "cosine", dtype, 9_000, dim, seed=4)
    ex, signs, offsets = _requests(stored, [3, 32, 2, 9], seed=5)
    _check(g, stored, "cosine", ex, signs, offsets, (10, 200), alone=(0, 2))
    g.close()


def test_more_than_32_requests_and_many_passes(G):
    g, stored = _gallery(G, "euclid", "bf16", 12_000, 64, seed=6)
    ex, signs, offsets = _requests(stored, [1] * 40 + [2] * 20 + [31], seed=7)
    _check(g, stored, "euclid", ex, signs, offsets, (7,), alone=(0, 39, 60))
    g.close()


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
def test_tie_cluster_forces_the_tighten_and_re_sweep(G, metric):
    """10 501 copies of one row: every copy ties at the top of a request whose positive is that row, more than the 8192
    rows a list holds, so the sweep overflows, tightens to the k-th (score, row) pair and sweeps again."""
    rng = np.random.default_rng(8)
    n, dim = 20_000, 96
    x = rng.standard_normal((n, dim)).astype(np.float32)
    x[rng.permutation(n)[:10_501]] = x[0]
    g = G(dim, dtype="f32", metric=metric, capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    is_copy = (stored == stored[0]).all(axis=1)
    other = stored[np.nonzero(~is_copy)[0][0]]
    ex = np.stack([stored[0], other, stored[0]])
    signs = np.array([1, -1, 1], np.int8)
    offsets = np.array([0, 2, 3])
    _check(g, stored, metric, ex, signs, offsets, (10, 1024), alone=(0,))
    res = g.recommend(ex, signs, offsets, 10)
    assert res.stats["fallback_queries"] > 0
    assert np.array_equal(res.rows[1], np.nonzero(is_copy)[0][:10])
    g.close()


def test_empty_requests_empty_gallery_and_device_inputs(G):
    import torch

    g = G(64, dtype="bf16", metric="cosine", capacity=16)
    res = g.recommend(np.zeros((0, 64), np.float32), np.zeros(0, np.int8), [0], 5)
    assert res.rows.shape == (0, 5)
    one = np.ones((2, 64), np.float32)
    res = g.recommend(one, [1, -1], [0, 2], 5, want_keys=True)
    assert np.all(res.rows == -1) and np.all(np.isneginf(res.scores)) and np.all(np.isneginf(res.scores64))
    g.close()
    g, stored = _gallery(G, "dot", "f16", 15_000, 200, seed=9)
    ex, signs, offsets = _requests(stored, [4, 1, 32, 6], seed=10)
    masks = _mask_set(len(stored), seed=11)
    words = np.stack([O.pack_row_mask(m) for m in masks])
    ids = np.array([3, -1, 2, 0], np.int32)
    host = g.recommend(ex, signs, offsets, 50, row_mask=words, mask_of_request=ids, want_keys=True)
    dev = g.recommend(torch.from_numpy(ex).cuda(), signs, offsets, 50, row_mask=torch.from_numpy(words.view(np.int32)).cuda(),
                      mask_of_request=torch.from_numpy(ids).cuda(), want_keys=True)
    assert dev.rows.is_cuda
    assert np.array_equal(dev.rows.cpu().numpy(), host.rows)
    assert np.array_equal(dev.scores64.cpu().numpy().view(np.uint64), host.scores64.view(np.uint64))
    shared = g.recommend(ex, signs, offsets, 50, row_mask=words[2], want_keys=True)   # one mask for every request
    _check(g, stored, "dot", ex, signs, offsets, (50,), masks[2:3], np.zeros(4, np.int32), alone=())
    assert np.array_equal(shared.rows, g.recommend(ex, signs, offsets, 50, row_mask=words[2:3],
                                                   mask_of_request=np.zeros(4, np.int32)).rows)
    g.close()


def test_client_recommend_on_a_real_gallery(tmp_path, monkeypatch):
    monkeypatch.setenv("RBOD_STORE_DIR", str(tmp_path))
    from qdrant_client import QdrantClient, models

    c = QdrantClient(location=":memory:")
    n, dim = 10_000, 48
    c.recreate_collection("r", vectors_config=models.VectorParams(size=dim, distance=models.Distance.COSINE))
    rng = np.random.default_rng(12)
    c.upsert("r", points=models.Batch(ids=list(range(n)), vectors=rng.standard_normal((n, dim)).astype(np.float32).tolist(),
                                      payloads=[{"class_name": f"c{i % 5}"} for i in range(n)]))
    col = c._root.get("r")
    stored = col.stored_vectors(range(n))
    flt = models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value="c2"))])
    got = c.recommend("r", positive=[10, 11], negative=[12], query_filter=flt, limit=7, strategy="best_score")
    allowed = np.array([i % 5 == 2 for i in range(n)])
    allowed[[10, 11, 12]] = False
    s, i = OR.recommend_topk(stored[[10, 11, 12]], [1, 1, -1], [0, 3], stored, 7, "cosine", [allowed])
    assert [p.id for p in got] == i[0].tolist()
    assert np.allclose([p.score for p in got], s[0], rtol=1e-7)
    reqs = [models.RecommendRequest(positive=[int(a), rng.standard_normal(dim).tolist()], negative=[int(b)] if j % 2 else None,
                                    filter=flt if j % 3 == 0 else None, limit=5, offset=j % 2, with_payload=True,
                                    strategy="best_score" if j % 2 else "average_vector")
            for j, (a, b) in enumerate(rng.integers(0, n, (12, 2)))]
    batch = c.recommend_batch("r", reqs)
    loop = [c.recommend("r", r.positive, r.negative, r.filter, r.limit, r.offset, strategy=r.strategy) for r in reqs]
    assert batch == loop and all(len(p) == 5 for p in batch)
    c.close()
