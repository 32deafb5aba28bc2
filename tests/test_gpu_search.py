"""K3 (tcgen05 cosine top-k) + exact rescoring through rbod_search, against the fp64 brute force."""
import numpy as np
import pytest

from oracle import oracle_c as OC
from oracle import oracle_np as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    from retrieval_based_object_detection_b200 import Gallery

    return Gallery


def _mk(G, n, dim, dtype, seed, clustered=False):
    if clustered:
        x, _, _ = O.synthetic_clustered(n, dim, max(2, n // 100), seed=seed)
    else:
        x = O.synthetic_unit_rows(n, dim, seed=seed)
    g = G(dim, dtype=dtype, capacity=n)
    g.upsert(x)
    return g, g.get_rows(np.arange(n)), x


RAW_SHAPES = [("bf16", 1000, 768, 130), ("f16", 200, 512, 5), ("f32", 513, 512, 128), ("bf16", 300, 64, 7),
              ("bf16", 4097, 320, 260)]
# the COSINE cases keep the ids they had before the metric became a parameter
RAW_CASES = [pytest.param(metric, *shape, id="-".join(map(str, shape)) + ("" if metric == "cosine" else "-" + metric))
             for metric in ("cosine", "dot", "euclid") for shape in RAW_SHAPES]


@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("metric,dtype,n,dim,Q", RAW_CASES)
def test_raw_tensor_core_scores(G, metric, variant, dtype, n, dim, Q):
    """The tcgen05 pass itself: q16 . g16 with fp32 accumulation, every (query, row) cell.  COSINE multiplies the unit
    query, DOT and EUCLID the query as given (rows and queries of different norms here), and EUCLID adds the row bias
    fp32(-|g|^2 / 2); fp32 galleries search an fp16 operand (COSINE) or a bf16 one (DOT, EUCLID)."""
    from test_gpu_gallery_lifecycle import raw_scores_reference

    x = O.synthetic_unit_rows(n, dim, seed=n)
    q = O.synthetic_unit_rows(Q, dim, seed=99)
    if metric != "cosine":
        x = x * np.linspace(0.25, 2.0, n, dtype=np.float32)[:, None]
        q = q * np.linspace(0.5, 1.5, Q, dtype=np.float32)[:, None]
    g = G(dim, dtype=dtype, metric=metric, capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    g.set_option("k3_variant", variant)
    got = g.debug_scores(q)
    want, tol = raw_scores_reference(metric, dtype, q, stored)
    assert got.shape == (Q, n) and not np.isnan(got).any()
    assert (np.abs(got - want) <= tol).all(), np.abs(got - want).max()
    g.close()


@pytest.mark.parametrize("dtype,dim", [("bf16", 1024), ("f16", 1280), ("f32", 2048)])
def test_wide_vectors_stay_on_the_tensor_cores(G, dtype, dim):
    """Rows wider than the TMEM-resident query tile allows (768 columns; e.g. 1024- and 1280-wide CLIP towers) run on
    the kernel flavour that streams the query tile through shared memory -- not on the fp64 sweep: raw tensor-core
    scores cell by cell, then ids identical to the brute force with no query left to the sweep."""
    n, Q, k = 40_000, 260, 10
    g, stored, x = _mk(G, n, dim, dtype, seed=dim)
    q = O.synthetic_unit_rows(Q, dim, seed=5)
    q[:100] = x[500:600] + 0.2 * O.synthetic_unit_rows(100, dim, seed=6)
    got = g.debug_scores(q[:9])
    kind = "bf16" if dtype == "bf16" else "f16"
    want = O.l2_normalize_store(q[:9], kind)[0].astype(np.float64) @ O.round_store(stored, kind).astype(np.float64).T
    assert np.abs(got - want).max() < 3e-5
    res = g.search(q, k, want_scores64=True)
    ws, wi = O.cosine_topk(q, stored, k)
    assert np.array_equal(res.rows, wi) and np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
    assert res.stats["k3_launches"] >= 1 and res.stats["sweep_queries"] == 0 and res.stats["candidates"] in (16, 32)
    g.close()


CASES = [
    # dtype, n, dim, Q, k, clustered
    ("f32", 1000, 512, 1000, 5, True),        # config C1 shape: 1k gallery, top-5
    ("bf16", 20000, 768, 300, 10, False),
    ("bf16", 20000, 768, 300, 100, False),
    ("f16", 5000, 768, 64, 10, True),
    ("f32", 30000, 512, 257, 10, True),
    ("bf16", 3, 512, 4, 10, False),           # fewer rows than k
    ("bf16", 64, 512, 1, 1, False),
    ("f32", 65, 100, 3, 40, False),           # dim not a multiple of 64 (padded operand)
    ("bf16", 150000, 768, 129, 10, False),    # many slices
]


@pytest.mark.parametrize("variant", [0, 2])
@pytest.mark.parametrize("dtype,n,dim,Q,k,clustered", CASES)
def test_search_matches_fp64_brute_force(G, variant, dtype, n, dim, Q, k, clustered):
    g, stored, x = _mk(G, n, dim, dtype, seed=n + k, clustered=clustered)
    g.set_option("k3_variant", variant)
    rng = np.random.default_rng(k)
    q = rng.standard_normal((Q, dim)).astype(np.float32)
    near = rng.integers(0, n, Q // 2)
    q[: Q // 2] = x[near] + 0.3 * q[: Q // 2] / np.sqrt(dim)       # queries close to stored rows
    res = g.search(q, k, want_scores64=True)
    ws, wi = O.cosine_topk(q, stored, k)
    assert np.array_equal(res.rows, wi), f"ids differ in {(res.rows != wi).any(axis=1).sum()} of {Q} queries"
    finite = np.isfinite(ws)
    assert np.allclose(res.scores64[finite], ws[finite], rtol=1e-5, atol=1e-9)      # tolerance of the north star
    assert np.array_equal(res.scores, res.scores64.astype(np.float32))
    assert np.all(np.isneginf(res.scores64[~finite]))
    assert res.stats["queries"] == Q and res.stats["k3_launches"] in (1, 2)
    g.close()


def test_duplicates_ties_and_fallback(G):
    """Exact duplicates tie; ties resolve to the smaller row slot; the certification fallback fires."""
    n, dim, k = 6000, 512, 10
    g, stored, x = _mk(G, n, dim, "bf16", seed=3)
    x2 = x.copy()
    x2[1000:1060] = x2[7]                    # 61 identical rows > kc: forces the exact fallback
    x2[2000] = x2[11]
    g.upsert(x2, slots=np.arange(n))
    stored = g.get_rows(np.arange(n))
    q = np.stack([x2[7] * 5.0, x2[11], x2[4000], -x2[7]]).astype(np.float32)
    res = g.search(q, k, want_scores64=True)
    ws, wi = OC.cosine_topk(q, stored, k)    # sequential C oracle: identical rows -> identical scores
    assert np.array_equal(res.rows, wi)
    assert list(res.rows[0]) == [7] + list(range(1000, 1009))
    assert list(res.rows[1][:2]) == [11, 2000]
    assert res.stats["fallback_queries"] >= 1
    assert np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
    g.close()


def test_wide_tie_cluster_goes_to_exact_sweep(G):
    """More identical rows than the collecting second pass records (1024): the fp64 sweep answers, its threshold
    seeded with the k-th exact score of the first pass -- in the key domain of each metric that can reach it."""
    n, dim, k = 9000, 512, 10
    x = O.synthetic_unit_rows(n, dim, seed=5)
    x[3000:4200] = x[17]                     # 1201 copies of row 17
    q = np.stack([x[17], x[5000]]).astype(np.float32)
    for metric in ("cosine", "dot", "euclid"):
        g = G(dim, dtype="bf16", metric=metric, capacity=n)
        g.upsert(x)
        stored = g.get_rows(np.arange(n))
        res = g.search(q, k, want_scores64=True)
        # sequential C oracle: identical rows -> identical scores
        ws, wi = OC.cosine_topk(q, stored, k) if metric == "cosine" else OC.distance_topk(q, stored, k, metric)
        assert np.array_equal(res.rows, wi), metric
        assert list(res.rows[0]) == [17] + list(range(3000, 3009)), metric
        assert np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9), metric
        assert res.stats["fallback_queries"] >= 1 and res.stats["sweep_queries"] >= 1, metric
        assert res.stats["k3_launches"] == 2, metric
        g.set_option("collect_pass", 0)      # the sweep alone gives the same answer
        res2 = g.search(q, k, want_scores64=True)
        assert np.array_equal(res2.rows, wi) and res2.stats["k3_launches"] == 1, metric
        assert res2.stats["sweep_queries"] >= 1, metric
        g.close()


def test_bf16_gallery_with_fp16_shadow_operand(G):
    """Option shadow16: a bf16 collection searched through an fp16 copy.  Stored rows, ids and scores are
    those of the bf16 gallery; the certification margin shrinks ~6x, so k=100 needs no second pass."""
    n, dim, Q, k = 120000, 768, 200, 100
    x = O.synthetic_unit_rows(n, dim, seed=21)
    x[5, :40] *= 1e-6                                    # elements far below fp16's normal range
    g = G(dim, dtype="bf16", capacity=n)
    g.set_option("shadow16", 1)
    g.upsert(x[: n // 2])
    g.upsert(x[n // 2:])                                 # second upsert grows nothing but appends to both copies
    stored = g.get_rows(np.arange(n))
    want_rows = O.l2_normalize_store(x, "bf16")[0]          # the stored rows stay bf16 (<= 1 bf16 ulp from the oracle)
    assert np.abs(stored.view(np.int32).astype(np.int64) - want_rows.view(np.int32).astype(np.int64)).max() <= 65536
    q = O.synthetic_unit_rows(Q, dim, seed=77)
    q[0] = x[5]
    res = g.search(q, k, want_scores64=True)
    ws, wi = O.cosine_topk(q, stored, k)
    assert np.array_equal(res.rows, wi)
    assert np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
    assert res.stats["max_eps"] < 6e-4 and res.stats["fallback_queries"] <= 2
    got = g.debug_scores(q[:4])                           # raw tensor-core scores come from the fp16 operand
    qn = O.l2_normalize_store(q[:4], "f16")[0].astype(np.float64)
    want = qn @ O.round_store(stored, "f16").astype(np.float64).T
    assert np.abs(got - want).max() < 2e-5
    from retrieval_based_object_detection_b200._native import RbodError
    with pytest.raises(RbodError):
        g.set_option("shadow16", 0)                       # only while the collection is empty
    g.close()


def test_bf16_gallery_builds_its_fp16_shadow_when_k_is_large(G):
    """A bf16 COSINE collection searched with k > 40 gets the fp16 search operand on the fly (one pass over the stored
    rows): the first k = 100 search is already certified with the small margin, rows upserted afterwards land in both
    copies, and the stored rows / ids / scores stay those of the bf16 gallery."""
    n, dim, Q, k = 120000, 768, 200, 100
    x = O.synthetic_unit_rows(n, dim, seed=21)
    x[5, :40] *= 1e-6                                    # elements far below fp16's normal range
    g = G(dim, dtype="bf16", capacity=n // 2)
    g.upsert(x[: n // 2])
    q = O.synthetic_unit_rows(Q, dim, seed=77)
    q[0] = x[5]
    r10 = g.search(q, 10)                                # k <= 40: plain bf16 operand
    assert r10.stats["max_eps"] > 1e-3
    stored_half = g.get_rows(np.arange(n // 2))
    res = g.search(q, k, want_scores64=True)             # builds the shadow
    ws, wi = O.cosine_topk(q, stored_half, k)
    assert np.array_equal(res.rows, wi) and np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
    assert res.stats["max_eps"] < 6e-4 and res.stats["fallback_queries"] <= 2
    g.upsert(x[n // 2:])                                 # grows the gallery: both copies follow
    stored = g.get_rows(np.arange(n))
    assert np.array_equal(stored[: n // 2], stored_half)
    for kk in (100, 10):
        res = g.search(q, kk, want_scores64=True)
        ws, wi = O.cosine_topk(q, stored, kk)
        assert np.array_equal(res.rows, wi) and np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
        assert res.stats["max_eps"] < 6e-4
    got = g.debug_scores(q[:4])                           # raw tensor-core scores now come from the fp16 operand
    qn = O.l2_normalize_store(q[:4], "f16")[0].astype(np.float64)
    assert np.abs(got - qn @ O.round_store(stored, "f16").astype(np.float64).T).max() < 2e-5
    g.close()


@pytest.mark.parametrize("tau_share", [0, 1])
def test_k100_bf16_uncertified_queries_take_the_collect_pass(G, tau_share):
    """bf16 rounding leaves little slack at k=100 (kc=128): a good share of the queries is not certified by
    the first pass; the collecting pass must return exactly the brute-force ids for them."""
    n, dim, Q, k = 120000, 768, 200, 100
    g, stored, x = _mk(G, n, dim, "bf16", seed=21)
    g.set_option("tau_share", tau_share)
    g.set_option("auto_shadow", 0)                       # stay on the bf16 operand: this test is about the second pass
    q = O.synthetic_unit_rows(Q, dim, seed=77)
    res = g.search(q, k, want_scores64=True)
    assert res.stats["fallback_queries"] > 0 and res.stats["k3_launches"] == 2
    ws, wi = O.cosine_topk(q, stored, k)
    assert np.array_equal(res.rows, wi), f"ids differ in {(res.rows != wi).any(axis=1).sum()} of {Q} queries"
    assert np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
    assert res.stats["sweep_queries"] == 0
    g.close()


@pytest.mark.parametrize("dtype,ordered", [("bf16", False), ("f32", True), ("f16", True)])
def test_threshold_prepass_keeps_the_answer_exact(G, dtype, ordered):
    """Galleries large enough for the sampled starting thresholds (>= 320 tiles), random and stored in class
    order (the adversarial layout for a sample): ids identical to the brute force, with and without it."""
    n, dim, Q, k = 60000, 256, 300, 10
    x, labels, _ = O.synthetic_clustered(n, dim, 40, seed=4)
    if ordered:
        x = x[np.argsort(labels, kind="stable")]
    g = G(dim, dtype=dtype, capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    rng = np.random.default_rng(1)
    q = x[rng.integers(0, n, Q)] + 0.2 * rng.standard_normal((Q, dim)).astype(np.float32) / np.sqrt(dim)
    mask = rng.random(n) < 0.5
    ws, wi = O.cosine_topk(q, stored, k)
    wms, wmi = O.cosine_topk(q, stored, k, row_mask=mask)
    for presample in (2, 0):                                    # 2 = forced (a 300-query batch would skip it)
        g.set_option("presample", presample)
        res = g.search(q, k, want_scores64=True)
        assert np.array_equal(res.rows, wi), (presample, (res.rows != wi).any(axis=1).sum())
        assert np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
        assert res.stats["total_launches"] >= (5 if presample else 3)      # pre-pass = K3 sample launch + tau_init
        resm = g.search(q, k, row_mask=O.pack_row_mask(mask), want_scores64=True)
        assert np.array_equal(resm.rows, wmi)
    g.close()


def test_prepass_threshold_too_high_is_retried(G):
    """Every sampled tile holds a copy of the query: the starting threshold equals the best score, fewer than k
    rows beat it, and the call must be redone without the pre-pass -- same exact answer."""
    n, dim, k = 60000, 256, 10
    x = O.synthetic_unit_rows(n, dim, seed=12)
    tiles = (n + 127) // 128
    for g_ in range(8):                                   # K3_SAMPLE_GROUPS one-tile groups, spread over the gallery
        x[(g_ * tiles // 8) * 128 + 5] = x[77]
    g = G(dim, dtype="bf16", capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    q = np.stack([x[77], x[1234]]).astype(np.float32)
    ws, wi = OC.cosine_topk(q, stored, k)
    res = g.search(q, k, want_scores64=True)                 # a 2-query batch skips the pre-pass on its own
    assert np.array_equal(res.rows, wi) and res.stats["presample_retries"] == 0
    g.set_option("presample", 2)
    res = g.search(q, k, want_scores64=True)
    assert np.array_equal(res.rows, wi)
    assert res.stats["presample_retries"] >= 1
    g.close()


def test_row_mask_and_zero_vectors(G):
    n, dim, k, Q = 5000, 768, 10, 40
    g, stored, x = _mk(G, n, dim, "bf16", seed=8)
    rng = np.random.default_rng(0)
    allowed = rng.random(n) < 0.3
    q = rng.standard_normal((Q, dim)).astype(np.float32)
    q[0] = 0.0                                # zero query: every score is 0 -> ids 0..k-1 of the allowed rows
    res = g.search(q, k, row_mask=O.pack_row_mask(allowed), want_scores64=True)
    ws, wi = O.cosine_topk(q, stored, k, row_mask=allowed)
    assert np.array_equal(res.rows, wi)
    assert np.all(allowed[res.rows])
    none = g.search(q[:3], k, row_mask=O.pack_row_mask(np.zeros(n, bool)))
    assert np.all(none.rows == -1)
    g.close()


def test_empty_gallery_bad_args_and_device_io(G):
    import torch

    from retrieval_based_object_detection_b200._native import RbodError

    g = G(512, dtype="bf16")
    r = g.search(np.ones((2, 512), np.float32), 3)
    assert np.all(r.rows == -1) and np.all(np.isneginf(r.scores))
    x = O.synthetic_unit_rows(3000, 512, seed=1)
    g.upsert(x)
    with pytest.raises(RbodError):
        g.search(x[:2], 0)
    stored = g.get_rows(np.arange(3000))
    r500 = g.search(x[:2], 500, want_scores64=True)          # beyond the tensor-core candidate lists: exact fp64 sweep
    ws5, wi5 = O.cosine_topk(x[:2], stored, 500, rowwise=True)
    assert np.array_equal(r500.rows, wi5) and np.allclose(r500.scores64, ws5, rtol=1e-9, atol=1e-12)
    assert r500.stats["sweep_queries"] == 2
    with pytest.raises(RbodError):
        g.search(x[:2], 2000)                # more than any path keeps
    with pytest.raises(ValueError):
        g.search(np.ones((2, 100), np.float32), 3)
    qd = torch.from_numpy(x[:50]).cuda()
    r = g.search(qd, 10, want_scores64=True)  # device in -> device out
    assert r.rows.is_cuda and r.scores.is_cuda
    ws, wi = O.cosine_topk(x[:50], stored, 10)
    assert np.array_equal(r.rows.cpu().numpy(), wi)
    assert np.array_equal(r.rows.cpu().numpy()[:, 0], np.arange(50))       # each row finds itself first
    g.close()


def test_full_size_properties(G):
    """BASELINE-scale shapes, checked through size-independent properties (no brute force)."""
    import torch

    n, dim, Q, k = 2_000_000, 768, 512, 10
    g = G(dim, dtype="bf16", capacity=n)
    gen = torch.Generator("cuda").manual_seed(0)
    for a in range(0, n, 500_000):
        g.upsert(torch.randn(500_000, dim, device="cuda", generator=gen))
    assert len(g) == n
    probe = torch.randint(0, n, (Q,), device="cuda", generator=gen)
    q = g.get_rows(probe)                                  # stored rows as queries
    r = g.search(q, k, want_scores64=True)
    rows, s64 = r.rows.cpu().numpy(), r.scores64.cpu().numpy()
    assert np.array_equal(rows[:, 0], probe.cpu().numpy())               # self match is rank 0 ...
    assert np.all(np.abs(s64[:, 0] - 1.0) < 1e-12)                        # ... with cosine 1
    assert np.all(np.diff(s64, axis=1) <= 0)                              # sorted descending
    assert np.all((rows >= 0) & (rows < n)) and all(len(set(rw)) == k for rw in rows)
    # idempotence / linearity in the query norm: scaling a query changes nothing
    r2 = g.search(q * 7.5, k, want_scores64=True)
    assert np.array_equal(r2.rows.cpu().numpy(), rows)
    # the reported scores are the exact cosines of the reported rows
    chk = g.get_rows(torch.from_numpy(rows[:8].reshape(-1)).cuda()).double().reshape(8, k, dim)
    qq = q[:8].double()
    cos = torch.einsum("qd,qkd->qk", qq, chk) / (qq.norm(dim=1, keepdim=True) * chk.norm(dim=2))
    assert np.allclose(cos.cpu().numpy(), s64[:8], rtol=1e-9, atol=1e-12)
    # spot-check one query against the brute force over the whole gallery (torch fp64 on device)
    allrows = torch.cat([g.get_rows(torch.arange(a, a + 250_000, device="cuda")).double() @ qq[0]
                         / (qq[0].norm() * g.get_rows(torch.arange(a, a + 250_000, device="cuda")).double().norm(dim=1))
                         for a in range(0, n, 250_000)])
    top = torch.topk(allrows, k)
    assert np.array_equal(np.sort(top.indices.cpu().numpy()), np.sort(rows[0]))
    g.close()


def _torch_topk_fp64(q, stored, k, chunk=250_000):
    """Independent check on device: plain torch float64 cosine + top-k (continuous random data: no exact ties,
    the tie rule itself is covered by the duplicate tests)."""
    import torch

    qq = q.double()
    qn = qq.norm(dim=1, keepdim=True)
    best_s = torch.zeros((q.shape[0], 0), dtype=torch.float64, device=q.device)
    best_i = torch.zeros((q.shape[0], 0), dtype=torch.int64, device=q.device)
    for a in range(0, stored.shape[0], chunk):
        g = stored[a:a + chunk].double()
        sc = (qq @ g.T) / (qn * g.norm(dim=1)[None, :])
        top = torch.topk(sc, min(k, sc.shape[1]), dim=1)
        s_all, i_all = torch.cat([best_s, top.values], 1), torch.cat([best_i, top.indices + a], 1)
        o = torch.topk(s_all, min(k, s_all.shape[1]), dim=1).indices
        best_s, best_i = torch.gather(s_all, 1, o), torch.gather(i_all, 1, o)
    return best_s, best_i


def test_config_c2_full_size_fp32_gallery(G):
    """BASELINE config C2: 1M x 512 fp32 gallery, 10k-query batch, exact top-10 -- every query checked against
    a torch float64 brute force on the device (ids identical, scores within 1e-5 relative)."""
    import torch

    n, dim, Q, k = 1_000_000, 512, 10_000, 10
    g = G(dim, dtype="f32", capacity=n)
    gen = torch.Generator("cuda").manual_seed(2)
    centres = torch.nn.functional.normalize(torch.randn(1000, dim, device="cuda", generator=gen), dim=1)
    for a in range(0, n, 250_000):      # clustered rows (class = row mod 1000), CLIP-like score range
        lab = torch.arange(a, a + 250_000, device="cuda") % 1000
        g.upsert(centres[lab] + 0.4 * torch.randn(250_000, dim, device="cuda", generator=gen) / dim ** 0.5)
    stored = g.get_rows(torch.arange(n, device="cuda"))
    q = centres[torch.randint(0, 1000, (Q,), device="cuda", generator=gen)] + \
        0.4 * torch.randn(Q, dim, device="cuda", generator=gen) / dim ** 0.5
    r = g.search(q, k, want_scores64=True)
    assert r.stats["sweep_queries"] == 0
    for a in range(0, Q, 2000):
        ws, wi = _torch_topk_fp64(q[a:a + 2000], stored, k)
        assert torch.equal(r.rows[a:a + 2000], wi), int((r.rows[a:a + 2000] != wi).any(dim=1).sum())
        assert torch.allclose(r.scores64[a:a + 2000], ws, rtol=1e-5, atol=1e-9)
    g.close()


def test_config_c3_delegates_then_centroid_search(G):
    """BASELINE config C3: per-class mean + renormalise over 1M labelled 768-d rows (10k classes, label-sorted
    through a row index), then query-vs-centroid top-5."""
    import torch

    n, dim, C, Q, k = 1_000_000, 768, 10_000, 10_000, 5
    g = G(dim, dtype="f32", capacity=n)
    gen = torch.Generator("cuda").manual_seed(3)
    centres = torch.nn.functional.normalize(torch.randn(C, dim, device="cuda", generator=gen), dim=1)
    labels = torch.randint(0, C, (n,), device="cuda", generator=gen)
    for a in range(0, n, 250_000):
        g.upsert(centres[labels[a:a + 250_000]] + 0.4 * torch.randn(250_000, dim, device="cuda", generator=gen) / dim ** 0.5)
    order = torch.argsort(labels, stable=True)
    offsets = torch.zeros(C + 1, dtype=torch.int64, device="cuda")
    offsets[1:] = torch.cumsum(torch.bincount(labels, minlength=C), 0)
    cent = g.segment_mean(offsets, row_idx=order)
    # float64 reference of compute_average (32:9-10) + stored (renormalised fp32) form, on device
    stored = g.get_rows(torch.arange(n, device="cuda"))
    sums = torch.zeros(C, dim, dtype=torch.float64, device="cuda").index_add_(0, labels, stored.double())
    mean32 = (sums / (offsets[1:] - offsets[:-1]).clamp(min=1)[:, None].double()).float()
    want = (mean32.double() / mean32.double().norm(dim=1, keepdim=True)).float()
    assert float((cent - want).abs().max()) <= 2e-7
    gc = G(dim, dtype="f32", capacity=C)
    gc.upsert(cent)
    q = stored[torch.randint(0, n, (Q,), device="cuda", generator=gen)]
    r = gc.search(q, k, want_scores64=True)
    ws, wi = _torch_topk_fp64(q, gc.get_rows(torch.arange(C, device="cuda")), k)
    assert torch.equal(r.rows, wi) and torch.allclose(r.scores64, ws, rtol=1e-5, atol=1e-9)
    g.close()
    gc.close()


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_dot_collection_search(G, dtype):
    """Distance.DOT (util/qdrant_manager.py:61-66 offers it): nothing is normalised, score = q . g on the stored
    rows, same exactness machinery.  (Third-party semantics: parity unpinned.)"""
    n, dim, Q, k = 30000, 512, 150, 10
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((n, dim)) * rng.uniform(0.2, 3.0, (n, 1))).astype(np.float32)
    g = G(dim, dtype=dtype, metric="dot", capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    assert np.array_equal(stored, O.round_store(x, dtype))              # stored as given (rounded to the dtype)
    q = (rng.standard_normal((Q, dim)) * rng.uniform(0.5, 20.0, (Q, 1))).astype(np.float32)
    res = g.search(q, k, want_scores64=True)
    sc = q.astype(np.float64) @ stored.astype(np.float64).T
    ws, wi = O.topk_from_scores(sc, k)
    assert np.array_equal(res.rows, wi), int((res.rows != wi).any(axis=1).sum())
    assert np.allclose(res.scores64, ws, rtol=1e-9, atol=1e-9)
    g.close()


# ------------------------------------------------------------------ K5: EUCLID / MANHATTAN
@pytest.mark.parametrize("metric", ["euclid", "manhattan"])
@pytest.mark.parametrize("dtype,n,dim", [("f32", 20000, 512), ("bf16", 9000, 768), ("f32", 3000, 100)])
def test_distance_collections_exact_topk(G, metric, dtype, n, dim):
    """Distance.EUCLID / Distance.MANHATTAN (util/qdrant_manager.py:61-66): vectors stored as given, distances in
    fp64 on the stored values, ascending, ties to the smaller row -- against the float64 oracle, including a
    duplicate cluster wider than k, a row mask, k larger than the gallery's allowed rows, and a gallery larger
    than the kernel's record buffer (sample pass + sweep).  (Third-party semantics: parity unpinned.)"""
    Q, k = 70, 10
    rng = np.random.default_rng(n + dim)
    x = (rng.standard_normal((n, dim)) * rng.uniform(0.5, 2.0, (n, 1))).astype(np.float32)
    x[100:130] = x[7]                                                    # 31 identical rows
    g = G(dim, dtype=dtype, metric=metric, capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    assert np.array_equal(stored, O.round_store(x, dtype))
    q = (rng.standard_normal((Q, dim)) * 1.3).astype(np.float32)
    q[0] = stored[7]                                                     # distance 0 to the duplicate cluster
    q[1] = stored[500] + np.float32(1e-3)
    res = g.search(q, k, want_scores64=True)
    wd, wi, wk = O.distance_topk(q, stored, k, metric)
    assert np.array_equal(res.rows, wi), int((res.rows != wi).any(axis=1).sum())
    assert list(res.rows[0]) == [7] + list(range(100, 109)) and np.all(res.scores[0] == 0)
    assert np.allclose(res.scores64, wk, rtol=1e-12, atol=1e-300)
    assert np.allclose(res.scores, wd.astype(np.float32), rtol=1e-6)
    assert np.all(np.diff(res.scores, axis=1) >= 0)                      # distances ascend
    # row mask: every 3rd row allowed; k beyond what is allowed pads with (+inf, -1)
    allowed = np.zeros(n, dtype=bool)
    allowed[::3] = True
    res_m = g.search(q[:9], 25, row_mask=O.pack_row_mask(allowed), want_scores64=True)
    _, wi_m, wk_m = O.distance_topk(q[:9], stored, 25, metric, row_mask=allowed)
    assert np.array_equal(res_m.rows, wi_m) and np.allclose(res_m.scores64, wk_m, rtol=1e-12, atol=1e-300)
    few = np.zeros(n, dtype=bool)
    few[[3, 11, 4000 % n]] = True
    res_f = g.search(q[:2], 5, row_mask=O.pack_row_mask(few))
    assert np.all(res_f.rows[:, 3:] == -1) and np.all(np.isinf(res_f.scores[:, 3:])) and np.all(res_f.rows[:, :3] >= 0)
    # delegate means of such a collection are not renormalised
    off = np.array([0, 50, 50, 300], np.int64)
    cent = g.segment_mean(off)
    want_c = O.segment_mean_renorm(stored, None, off, normalize=False)
    assert np.all(cent[1] == 0) and np.allclose(cent, want_c, rtol=1e-6, atol=1e-7)
    g.close()


def test_distance_collection_device_io_and_empty(G):
    import torch

    g = G(64, dtype="f32", metric="euclid", capacity=16)
    r0 = g.search(np.zeros((2, 64), np.float32), 3)
    assert np.all(r0.rows == -1) and np.all(np.isinf(r0.scores))
    x = torch.randn(5000, 64, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    g.upsert(x)
    q = torch.randn(33, 64, device="cuda", generator=torch.Generator("cuda").manual_seed(2))
    r = g.search(q, 4, want_scores64=True)
    assert r.rows.is_cuda
    d = torch.cdist(q.double(), x.double())
    top = torch.topk(d, 4, dim=1, largest=False)
    assert torch.equal(top.indices, r.rows) and torch.allclose(top.values, r.scores.double(), rtol=1e-6)
    g.close()


@pytest.mark.parametrize("dtype,dim", [("bf16", 768), ("f16", 512), ("bf16", 320)])
def test_stage_width_and_split_prepass_do_not_change_the_answer(G, dtype, dim):
    """The planner's choices are invisible in the result: 2 or 4 k-blocks per pipeline stage (k3_kbs), the threshold
    pre-pass with its combs split over many CTAs (a gallery of >= 1024 tiles gives every sample group >= 2 tiles),
    forced on, off, or left to the batch-size rule -- always the ids of the float64 brute force."""
    n, Q, k = 140_000, 130, 10
    x = O.synthetic_unit_rows(n, dim, seed=31)
    g = G(dim, dtype=dtype, capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    q = O.synthetic_unit_rows(Q, dim, seed=32)
    q[:20] = x[1000:1020] + 0.05 * O.synthetic_unit_rows(20, dim, seed=33)
    ws, wi = O.cosine_topk(q, stored, k)
    seen = set()
    for kbs in (2, 4, 0):
        for presample in (2, 0, 1):
            g.set_option("k3_kbs", kbs)
            g.set_option("presample", presample)
            res = g.search(q, k, want_scores64=True)
            assert np.array_equal(res.rows, wi), (kbs, presample, int((res.rows != wi).any(axis=1).sum()))
            assert np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
            seen.add(res.stats["total_launches"])
    assert len(seen) >= 2                                   # with and without the two pre-pass launches
    res8 = g.search(q[:8], k)                               # <= 8 queries: the rule skips the pre-pass
    res9 = g.search(q[:9], k)
    assert res9.stats["total_launches"] == res8.stats["total_launches"] + 2
    assert np.array_equal(res8.rows, wi[:8]) and np.array_equal(res9.rows, wi[:9])
    g.close()


def _torch_topk_fp64_from_gallery(g, n, q, k, chunk=500_000):
    """Like _torch_topk_fp64, but pulls the stored rows out of the gallery chunk by chunk (a 10M x 768 gallery
    widened to float32 would not be worth holding twice)."""
    import torch

    qq = q.double()
    qq = qq / qq.norm(dim=1, keepdim=True)
    best_s = torch.zeros((q.shape[0], 0), dtype=torch.float64, device=q.device)
    best_i = torch.zeros((q.shape[0], 0), dtype=torch.int64, device=q.device)
    for a in range(0, n, chunk):
        rows = g.get_rows(torch.arange(a, min(a + chunk, n), device=q.device)).double()
        sc = (qq @ rows.T) / rows.norm(dim=1)[None, :]
        top = torch.topk(sc, min(k, sc.shape[1]), dim=1)
        s_all, i_all = torch.cat([best_s, top.values], 1), torch.cat([best_i, top.indices + a], 1)
        o = torch.topk(s_all, min(k, s_all.shape[1]), dim=1).indices
        best_s, best_i = torch.gather(s_all, 1, o), torch.gather(i_all, 1, o)
        del rows, sc
    return best_s, best_i


@pytest.mark.parametrize("dtype,n,Q,k", [("bf16", 10_000_000, 1024, 100),      # BASELINE config C4, one GPU's view
                                         ("f16", 12_500_000, 48, 10)])         # config C5: one GPU's 12.5M-row shard
def test_configs_c4_c5_full_size_exact(G, dtype, n, Q, k):
    """The 768-wide BASELINE configs at their full per-GPU size: every query against a torch float64 brute force
    over the stored rows (ids identical, scores within 1e-5 relative), plus the single-query latency path."""
    import torch

    dim = 768
    g = G(dim, dtype=dtype, capacity=n)
    gen = torch.Generator("cuda").manual_seed(17)
    for a in range(0, n, 500_000):
        g.upsert(torch.randn(min(500_000, n - a), dim, device="cuda", generator=gen))
    assert len(g) == n
    q = torch.randn(Q, dim, device="cuda", generator=gen)
    r = g.search(q, k, want_scores64=True)
    ws, wi = _torch_topk_fp64_from_gallery(g, n, q, k)
    assert torch.equal(r.rows, wi), int((r.rows != wi).any(dim=1).sum())
    assert torch.allclose(r.scores64, ws, rtol=1e-5, atol=1e-9)
    assert r.stats["sweep_queries"] == 0
    r1 = g.search(q[:1], k, want_scores64=True)               # Q = 1: the HBM-bound end of the C5 sweep
    assert torch.equal(r1.rows, wi[:1])
    g.close()


@pytest.mark.parametrize("dtype", ["f32", "bf16", "f16"])
def test_euclid_collection_on_the_tensor_core_path(G, dtype):
    """EUCLID collections up to 768 columns run on the tcgen05 pass with the row-bias epilogue (score = q.g - |g|^2/2),
    exact rescoring of -|q-g|^2 in fp64 and the usual certification: a mid-size gallery of rows with very different
    norms, every query against torch.cdist in float64 (ids identical, distances within 1e-6 relative)."""
    import torch

    n, dim, Q, k = 300_000, 512, 1500, 10
    gen = torch.Generator("cuda").manual_seed(41)
    x = torch.randn(n, dim, device="cuda", generator=gen) * (0.05 + 2.0 * torch.rand(n, 1, device="cuda", generator=gen))
    if dtype == "f16":
        x = x * 0.25
    g = G(dim, dtype=dtype, metric="euclid", capacity=1000)          # grows several times: the bias array follows
    for a in range(0, n, 100_000):
        g.upsert(x[a:a + 100_000])
    stored = g.get_rows(torch.arange(n, device="cuda"))
    q = torch.randn(Q, dim, device="cuda", generator=gen) * (0.1 + torch.rand(Q, 1, device="cuda", generator=gen))
    q[:50] = stored[1000:1050] + 0.01 * torch.randn(50, dim, device="cuda", generator=gen)   # near neighbours exist
    r = g.search(q, k, want_scores64=True)
    assert r.stats["k3_launches"] >= 1 and r.stats["sweep_queries"] < Q           # tensor-core path, not the K5 sweep
    d = torch.cdist(q.double(), stored.double())
    top = torch.topk(d, k, dim=1, largest=False)
    assert torch.equal(top.indices, r.rows), int((top.indices != r.rows).any(dim=1).sum())
    assert torch.allclose(top.values, r.scores.double(), rtol=1e-6, atol=1e-9)
    assert torch.allclose(-top.values ** 2, r.scores64, rtol=1e-9, atol=1e-12)
    # overwrite a row: its bias follows
    g.upsert(q[7:8], slots=np.array([123], dtype=np.int64))
    r2 = g.search(q[7:8], 3)
    assert int(r2.rows[0, 0]) == 123 and float(r2.scores[0, 0]) <= (0.0 if dtype == "f32" else 1e-1)
    g.close()


def test_refused_cooperative_launch_falls_back_to_a_plain_grid(G):
    """The L2-sharing throttle makes CTAs of one launch wait for each other, so it asks for a cooperative launch; when
    the runtime refuses (the grid cannot be co-resident: fewer SMs than planned) the search must drop the throttle and
    run as an ordinary grid -- same exact answer, no error, no poisoned context.  The test hook over-sizes the grid
    (2 CTAs per SM with one resident), which makes the runtime refuse."""
    n, dim, Q, k = 150_000, 768, 129, 10                 # several slices x 2 query tiles: the throttle is in play
    g, stored, x = _mk(G, n, dim, "bf16", seed=9)
    q = O.synthetic_unit_rows(Q, dim, seed=10)
    ws, wi = O.cosine_topk(q, stored, k)
    res = g.search(q, k, want_scores64=True)
    assert np.array_equal(res.rows, wi) and g.info()["coop_refusals"] == 0
    g.set_option("debug_grid_scale", 2)
    res = g.search(q, k, want_scores64=True)
    assert np.array_equal(res.rows, wi) and np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
    assert g.info()["coop_refusals"] >= 1
    g.set_option("debug_grid_scale", 1)
    res = g.search(q, k)
    assert np.array_equal(res.rows, wi)                  # and the collection keeps working
    g.close()


def test_upsert_accepts_device_resident_slots(G):
    """include/rbod.h: row_slots may live on the host or on the device."""
    import torch

    g = G(64, dtype="f32", capacity=16)
    x = torch.randn(8, 64, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    g.upsert(x)
    y = torch.randn(2, 64, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    slots = torch.tensor([5, 8], dtype=torch.int64, device="cuda")      # overwrite row 5, append row 8
    import ctypes

    from retrieval_based_object_detection_b200 import _native as N

    N.check(g._lib.rbod_upsert(g._h, y.data_ptr(), 2, slots.data_ptr(), None, 0, None))
    torch.cuda.synchronize()
    assert len(g) == 9
    rows = g.get_rows(torch.tensor([5, 8], device="cuda"))
    assert torch.allclose(rows, y / y.norm(dim=1, keepdim=True), atol=1e-6)
    g.close()


@pytest.mark.parametrize("dtype", ["bf16", "f32"])
def test_tie_cluster_wider_than_the_sweep_list_still_answers(G, dtype):
    """More identical rows than even the exact sweep records per query (8192) -- the same image upserted under many
    ids, or a block of all-equal vectors: the search used to fail with RBOD_E_OVERFLOW.  The sweep now tightens an
    overflowing list to the k-th best (score, row) pair it did record and sweeps again, so the answer is the k
    smallest row slots of the tie, exactly as the (score desc, id asc) order says."""
    n, dim = 20_000, 256
    x = O.synthetic_unit_rows(n, dim, seed=77)
    x[3000:13500] = x[17]                                  # 10501 copies of row 17
    g = G(dim, dtype=dtype, capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    q = np.stack([x[17], x[15000], x[17] + 0.01 * x[15000]]).astype(np.float32)
    for k in (10, 100):
        res = g.search(q, k, want_scores64=True)
        ws, wi = OC.cosine_topk(q, stored, k)              # sequential C oracle: identical rows -> identical scores
        assert np.array_equal(res.rows, wi), (k, int((res.rows != wi).any(axis=1).sum()))
        assert list(res.rows[0][:4]) == [17, 3000, 3001, 3002]
        assert np.allclose(res.scores64, ws, rtol=1e-5, atol=1e-9)
        assert res.stats["sweep_queries"] >= 1
    mask = np.ones(n, dtype=bool)
    mask[3000:3050] = False                                # with a row mask the tie starts later
    res = g.search(q[:1], 10, row_mask=O.pack_row_mask(mask))
    assert list(res.rows[0]) == [17] + list(range(3050, 3059))
    g.close()


@pytest.mark.parametrize("metric,k", [("manhattan", 10), ("cosine", 200)])
def test_k5_tie_cluster_wider_than_its_lists(G, metric, k):
    """The fp64 sweep (MANHATTAN, or k beyond the tensor-core lists) with more identical rows than its 8192-entry
    lists hold: overflowing lists are tightened to the k-th best (key, row) pair, so the k smallest row slots of the
    tie come back instead of RBOD_E_OVERFLOW."""
    n, dim = 13_000, 64
    rng = np.random.default_rng(5)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    x[1000:11500] = x[7]                                   # 10501 copies of row 7
    g = G(dim, dtype="f32", metric=metric, capacity=n)
    g.upsert(x)
    stored = g.get_rows(np.arange(n))
    q = np.stack([x[7], x[12000]]).astype(np.float32)
    res = g.search(q, k, want_scores64=True)
    if metric == "cosine":
        ws, wi = OC.cosine_topk(q, stored, k)
    else:
        ws, wi, _ = O.distance_topk(q, stored, k, metric)
    assert np.array_equal(res.rows, wi), int((res.rows != wi).any(axis=1).sum())
    assert list(res.rows[0][:3]) == [7, 1000, 1001]
    assert res.stats["sweep_queries"] == 2
    g.close()
