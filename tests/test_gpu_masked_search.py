"""rbod_search_masks: one row mask per query, answered in one pass, against the fp64 oracle run once per mask with
that mask, and bit for bit against one rbod_search per query."""
import numpy as np
import pytest

from oracle import oracle_c as OC
from oracle import oracle_np as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    from retrieval_based_object_detection_b200 import Gallery

    return Gallery


def _oracle(q, stored, k, metric, allowed):
    if metric == "cosine":
        return OC.cosine_topk(q, stored, k, row_allowed=allowed)
    return OC.distance_topk(q, stored, k, metric, row_allowed=allowed)


def _mask_set(n, k, seed):
    """Masks that allow nothing, one row, fewer than k rows, 1 %, 30 % and every row."""
    rng = np.random.default_rng(seed)
    m = np.zeros((6, n), dtype=bool)
    m[1, rng.integers(0, n)] = True
    m[2, rng.choice(n, max(1, k // 2), replace=False)] = True
    m[3] = rng.random(n) < 0.01
    m[4] = rng.random(n) < 0.30
    m[5] = True
    return m


def _ids(Q, n_masks, seed):
    """Every mask and -1 (no filter), mixed."""
    ids = np.arange(Q, dtype=np.int32) % (n_masks + 1) - 1
    return np.random.default_rng(seed).permutation(ids).astype(np.int32)


def _check(g, stored, q, k, metric, masks, ids, per_query=None, **kw):
    """Ids identical to the oracle, fp64 scores within the search tests' tolerance, and (for the queries in
    ``per_query``) every output bit equal to one rbod_search with the query's own mask."""
    words = np.stack([O.pack_row_mask(m) for m in masks])
    res = g.search(q, k, row_mask=words, mask_of_query=ids, want_scores64=True, **kw)
    for mid in np.unique(ids):
        sel = np.nonzero(ids == mid)[0]
        ws, wi = _oracle(q[sel], stored, k, metric, None if mid < 0 else masks[mid])
        assert np.array_equal(res.rows[sel], wi), (int(mid), int((res.rows[sel] != wi).any(axis=1).sum()))
        finite = np.isfinite(ws)
        assert np.allclose(res.scores64[sel][finite], ws[finite], rtol=1e-5, atol=1e-9), int(mid)
        assert np.all(res.rows[sel][~finite] == -1)
        if mid >= 0:
            got = res.rows[sel]
            assert np.all(masks[mid][got[got >= 0]])
    for i in (range(len(q)) if per_query is None else per_query):
        one = g.search(q[i:i + 1], k, row_mask=None if ids[i] < 0 else words[ids[i]], want_scores64=True)
        assert np.array_equal(one.rows[0], res.rows[i]), i
        assert np.array_equal(one.scores[0].view(np.uint32), res.scores[i].view(np.uint32)), i
        assert np.array_equal(one.scores64[0].view(np.uint64), res.scores64[i].view(np.uint64)), i
    return res


def _gallery(G, metric, dtype, n, dim, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    if metric != "cosine":
        x *= rng.uniform(0.2, 2.0, (n, 1)).astype(np.float32)
    g = G(dim, dtype=dtype, metric=metric, capacity=n)
    g.upsert(x)
    return g, g.get_rows(np.arange(n)), x


@pytest.mark.parametrize("metric", ["cosine", "dot", "euclid"])
@pytest.mark.parametrize("dtype", ["bf16", "f16", "f32"])
def test_per_query_masks_match_the_oracle(G, metric, dtype):
    """Every mask kind mixed with unfiltered queries, on each kernel flavour: the single-CTA kernel with Q = 5 (no
    pre-pass), the streamed query tile with Q = 100, CTA pairs with Q = 300."""
    n, dim, k = 20_000, 256, 10
    g, stored, x = _gallery(G, metric, dtype, n, dim, seed=len(metric) + len(dtype))
    masks = _mask_set(n, k, seed=3)
    rng = np.random.default_rng(9)
    for variant, Q in ((0, 5), (1, 100), (2, 300)):
        g.set_option("k3_variant", variant)
        q = rng.standard_normal((Q, dim)).astype(np.float32)
        q[: Q // 2] = x[rng.integers(0, n, Q // 2)] + 0.3 * q[: Q // 2] / np.sqrt(dim)
        ids = _ids(Q, len(masks), seed=Q)
        res = _check(g, stored, q, k, metric, masks, ids, per_query=range(min(Q, 24)))
        assert res.stats["queries"] == Q and res.stats["sweep_queries"] < Q
    g.close()


def test_wide_rows_on_the_streamed_flavour(G):
    n, dim, Q, k = 8000, 1024, 140, 10
    g, stored, x = _gallery(G, "cosine", "bf16", n, dim, seed=1)
    masks = _mask_set(n, k, seed=4)
    q = O.synthetic_unit_rows(Q, dim, seed=2)
    _check(g, stored, q, k, "cosine", masks, _ids(Q, len(masks), seed=1), per_query=range(16))
    g.close()


def test_prepass_with_class_masks(G):
    """60 000 rows stored in class order, the pre-pass forced, every query filtered to one class: each query's starting
    threshold comes from its own class.  Then the case of test_prepass_threshold_too_high_is_retried with per-query
    masks: the pre-pass is retried and the answer stays exact."""
    n, dim, Q, k = 60_000, 256, 300, 10
    x, labels, _ = O.synthetic_clustered(n, dim, 40, seed=4)
    order = np.argsort(labels, kind="stable")
    x, labels = x[order], labels[order]
    g = G(dim, dtype="bf16", capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    g.set_option("presample", 2)
    masks = np.stack([labels == c for c in range(40)])
    rng = np.random.default_rng(1)
    q = x[rng.integers(0, n, Q)] + 0.2 * rng.standard_normal((Q, dim)).astype(np.float32) / np.sqrt(dim)
    ids = rng.integers(0, 40, Q).astype(np.int32)
    res = _check(g, stored, q, k, "cosine", masks, ids, per_query=range(8))
    assert res.stats["total_launches"] >= 5                      # K3 sample launch + tau_init ran
    g.close()

    x = O.synthetic_unit_rows(n, dim, seed=12)
    tiles = (n + 127) // 128
    for g_ in range(8):
        x[(g_ * tiles // 8) * 128 + 5] = x[77]
    g = G(dim, dtype="bf16", capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    g.set_option("presample", 2)
    q = np.stack([x[77], x[1234], x[77], x[1234]]).astype(np.float32)
    masks = np.ones((2, n), dtype=bool)
    masks[1, n // 2:] = False
    res = _check(g, stored, q, k, "cosine", masks, np.array([0, 0, 1, -1], dtype=np.int32))
    assert res.stats["presample_retries"] >= 1
    g.close()


@pytest.mark.parametrize("collect_pass", [1, 0])
def test_tie_cluster_collecting_pass_and_sweep(G, collect_pass):
    """1201 copies of one row leave the queries aimed at it uncertified.  Some of them may see the copies, others
    have them masked out: the gathered rows of the collecting pass and the sweep's batch slots must carry each query's
    own mask."""
    n, dim, k = 9000, 512, 10
    x = O.synthetic_unit_rows(n, dim, seed=5)
    x[3000:4200] = x[17]
    g = G(dim, dtype="bf16", capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    g.set_option("collect_pass", collect_pass)
    masks = np.ones((3, n), dtype=bool)
    masks[0, 3000:4200] = False                   # the copies masked out
    masks[1, 3000:3600] = False                   # half of them masked out
    masks[2, ::2] = False
    q = np.stack([x[17], x[17], x[17], x[17], x[5000], x[17] + 0.001 * x[5000]] * 7).astype(np.float32)
    ids = np.array([-1, 0, 1, 2, 1, 0] * 7, dtype=np.int32)
    res = _check(g, stored, q, k, "cosine", masks, ids, per_query=range(6))
    assert res.stats["fallback_queries"] > 0 and res.stats["sweep_queries"] > 0
    g.close()


@pytest.mark.parametrize("metric,dim,k", [("manhattan", 256, 10), ("cosine", 256, 200), ("euclid", 2304, 10)])
def test_k5_sweep_with_mixed_masks_per_batch(G, metric, dim, k):
    """The direct K5 sweep (MANHATTAN, k > 128, rows wider than 2048) with 70 queries: every 32-query batch mixes
    masks and unfiltered slots."""
    n, Q = 6000, 70
    g, stored, x = _gallery(G, metric, "f32", n, dim, seed=dim + k)
    masks = _mask_set(n, k, seed=5)
    q = np.random.default_rng(6).standard_normal((Q, dim)).astype(np.float32)
    res = _check(g, stored, q, k, metric, masks, _ids(Q, len(masks), seed=7), per_query=range(10))
    assert res.stats["sweep_queries"] == Q
    g.close()


def test_device_inputs_errors_and_edge_cases(G):
    import torch

    from retrieval_based_object_detection_b200._native import RBOD_E_INVAL, RbodError

    n, dim, Q, k = 5000, 256, 40, 10
    g, stored, x = _gallery(G, "cosine", "bf16", n, dim, seed=11)
    masks = _mask_set(n, k, seed=8)
    words = np.stack([O.pack_row_mask(m) for m in masks])
    ids = _ids(Q, len(masks), seed=3)
    q = O.synthetic_unit_rows(Q, dim, seed=4)
    host = g.search(q, k, row_mask=words, mask_of_query=ids, want_scores64=True)
    dev = g.search(torch.from_numpy(q).cuda(), k, row_mask=torch.from_numpy(words.view(np.int32)).cuda(),
                   mask_of_query=torch.from_numpy(ids).cuda(), want_scores64=True)
    assert torch.equal(dev.rows.cpu(), torch.from_numpy(host.rows))
    assert torch.equal(dev.scores64.cpu(), torch.from_numpy(host.scores64))
    # mask_of_query = None: every query reads mask 0, as rbod_search with that mask
    shared = g.search(q, k, row_mask=words[4:5], mask_of_query=None, want_scores64=True)
    plain = g.search(q, k, row_mask=words[4], want_scores64=True)
    assert np.array_equal(shared.rows, plain.rows) and np.array_equal(shared.scores64, plain.scores64)
    all_minus1 = g.search(q, k, row_mask=words, mask_of_query=np.full(Q, -1, np.int32), want_scores64=True)
    unfiltered = g.search(q, k, want_scores64=True)
    assert np.array_equal(all_minus1.rows, unfiltered.rows)
    lib = g._lib
    for bad in (len(masks), -2):
        b = ids.copy()
        b[3] = bad
        with pytest.raises(RbodError) as e:
            g.search(q, k, row_mask=words, mask_of_query=b)
        assert e.value.code == RBOD_E_INVAL
    out_s = np.empty((Q, k), np.float32)
    out_r = np.empty((Q, k), np.int64)
    rc = lib.rbod_search_masks(g._h, q.ctypes.data, Q, k, None, 2, ids.ctypes.data, out_s.ctypes.data,
                               out_r.ctypes.data, None, None, None)
    assert rc == RBOD_E_INVAL
    rc = lib.rbod_search_masks(g._h, q.ctypes.data, Q, k, words.ctypes.data, -1, None, out_s.ctypes.data,
                               out_r.ctypes.data, None, None, None)
    assert rc == RBOD_E_INVAL
    # Q = 0 and an empty gallery behave as rbod_search
    z = g.search(q[:0], k, row_mask=words, mask_of_query=ids[:0])
    assert z.rows.shape == (0, k)
    g.close()
    e = G(dim, dtype="bf16")
    r = e.search(q[:3], k, row_mask=np.zeros((2, 0), np.uint32), mask_of_query=np.array([0, -1, 1], np.int32))
    assert np.all(r.rows == -1) and np.all(np.isneginf(r.scores))
    e.close()


def test_client_search_batch_equals_the_request_loop(store_dir):
    from qdrant_client import QdrantClient, models

    c = QdrantClient(host="localhost", port=6333)
    n, dim = 3000, 64
    rng = np.random.default_rng(2)
    vecs = rng.standard_normal((n, dim)).astype(np.float32)
    c.recreate_collection("b", vectors_config=models.VectorParams(size=dim, distance=models.Distance.COSINE))
    c.upsert("b", points=models.Batch(ids=list(range(n)), vectors=vecs.tolist(),
                                      payloads=[{"class_name": f"c{i % 7}", "seg": i % 3 == 0} for i in range(n)]))
    flts = [None] + [models.Filter(must=[models.FieldCondition(key="class_name", match=models.MatchValue(value=f"c{j}"))])
                     for j in range(7)] + [models.Filter(must_not=[models.FieldCondition(key="seg",
                                                                                          match=models.MatchValue(value=True))])]
    reqs = [models.SearchRequest(vector=rng.standard_normal(dim).tolist(), filter=flts[i % len(flts)],
                                 limit=(5, 10, 20)[i % 3], offset=i % 2, with_payload=i % 2 == 0,
                                 score_threshold=0.05 if i % 5 == 0 else None) for i in range(60)]
    got = c.search_batch("b", requests=reqs)
    want = [c.search("b", r.vector, r.filter, r.limit, r.offset, bool(r.with_payload), bool(r.with_vector),
                     r.score_threshold) for r in reqs]
    assert got == want
    c.close()
