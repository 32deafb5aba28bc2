"""Galleries after they are built: overwrites, growth, RAW moves, truncation, deletes, option changes and reloads.

Every derived buffer of a collection (fp32 master, 16-bit search operand, fp16 shadow, EUCLID row bias, the `stats`
maxima behind the certification margin) has to follow each mutation, and rows that a truncate forgot keep their bytes
in every buffer without ever being seen again.  The checks run against a numpy model of the rows that should be
present, with the fp64 oracle of test_gpu_fuzz.py."""
import shutil

import numpy as np
import pytest

from oracle import oracle_np as O
from test_gpu_fuzz import _want

pytestmark = pytest.mark.gpu

METRICS = ("cosine", "dot", "euclid", "manhattan")
DTYPES = ("f32", "bf16", "f16")
DIMS = (100, 256, 768)


def _operand_kind(metric, dtype, shadow):
    """16-bit type of the tensor-core operands: fp16 for f16 stores, fp32 COSINE masters and the bf16 shadow."""
    return "f16" if dtype == "f16" or shadow or (dtype == "f32" and metric == "cosine") else "bf16"


def raw_scores_reference(metric, dtype, q, stored, shadow=False):
    """What rbod_debug_scores must return, in fp64, and the per-cell tolerance: q16 . g16 (+ fp32(-|g|^2 / 2) for
    EUCLID), q16 = the unit query (COSINE) or the query itself, g16 = the stored rows, both rounded to the operand type.
    Tolerance: fp32 accumulation, 2e-5 |q16| |g16|, plus the rounding of the bias addition."""
    kind = _operand_kind(metric, dtype, shadow)
    q16 = (O.l2_normalize_store(q, kind)[0] if metric == "cosine" else O.round_store(q, kind)).astype(np.float64)
    g16 = O.round_store(stored, kind).astype(np.float64)
    dots = q16 @ g16.T
    tol = 2e-5 * np.linalg.norm(q16, axis=1)[:, None] * np.linalg.norm(g16, axis=1)[None, :]
    if metric != "euclid":
        return dots, tol
    s64 = stored.astype(np.float64)
    bias = (-0.5 * np.einsum("ij,ij->i", s64, s64)).astype(np.float32).astype(np.float64)
    return dots + bias[None, :], tol + 1.2e-7 * (np.abs(dots) + np.abs(bias)[None, :])


def _storage_ulps(a, b, dtype):
    """Largest difference in units of the storage type's last place (both arrays hold values of that type)."""
    if dtype == "f16":
        ia, ib = a.astype(np.float16).view(np.int16), b.astype(np.float16).view(np.int16)
    else:
        ia, ib = a.view(np.int32) >> (16 if dtype == "bf16" else 0), b.view(np.int32) >> (16 if dtype == "bf16" else 0)
    return int(np.abs(ia.astype(np.int64) - ib.astype(np.int64)).max()) if a.size else 0


class _Model:
    """The rows a gallery should hold: per slot, what get_rows returned right after the slot was written."""

    def __init__(self, g, metric, dtype, dim):
        self.g, self.metric, self.dtype, self.dim = g, metric, dtype, dim
        self.rows = np.zeros((0, dim), np.float32)
        self.forgotten = []        # stored vectors that were truncated away or moved out of their slot
        self.shadow = False
        self.capacities = set()

    def wrote(self, slots, inputs, raw=False):
        """Reads back freshly written slots, checks them against the oracle's stored form (K1 tolerance) unless they
        are RAW copies of stored rows (then bit for bit), and records them."""
        slots = np.asarray(slots, np.int64)
        n = max(len(self.rows), int(slots.max()) + 1)
        if n > len(self.rows):
            self.rows = np.concatenate([self.rows, np.zeros((n - len(self.rows), self.dim), np.float32)])
        got = self.g.get_rows(slots)
        if raw:
            assert np.array_equal(got, inputs)
        else:
            want = (O.l2_normalize_store(inputs, self.dtype)[0] if self.metric == "cosine"
                    else O.round_store(inputs, self.dtype))
            assert _storage_ulps(got, want, self.dtype) <= 1
            assert np.count_nonzero(got != want) <= max(2, 1e-4 * got.size)
        self.rows[slots] = got

    def truncate(self, rows):
        self.forgotten.extend(self.rows[rows:])
        self.rows = self.rows[:rows].copy()
        self.g.truncate(rows)


def _rand_rows(rng, m, dim, metric):
    scale = rng.uniform(0.3, 1.5, (m, 1)) * (1.0 if metric == "cosine" else 0.5)
    return (rng.standard_normal((m, dim)) * scale).astype(np.float32)


def _upsert_device_slots(g, rows, slots):
    """rbod_upsert with the slot array in device memory (Gallery.upsert always passes host slots)."""
    import torch

    from retrieval_based_object_detection_b200 import _native as N

    r = torch.as_tensor(rows, device="cuda").float().contiguous()
    s = torch.as_tensor(np.asarray(slots, np.int64), device="cuda").contiguous()
    N.check(g._lib.rbod_upsert(g._h, r.data_ptr(), r.shape[0], s.data_ptr(), None, 0, None))
    torch.cuda.synchronize()


def _check_search(res, k, want, n_rows):
    """Ids equal to the oracle's first k (its lists are ordered, so a longer list serves every smaller k), fp64
    scores within test_gpu_fuzz.py's tolerance, no slot at or beyond the row count."""
    _, wi, wk = want
    wi, wk = wi[:, :k], wk[:, :k]
    assert np.array_equal(res.rows, wi), (k, int((res.rows != wi).any(axis=1).sum()))
    fin = wi >= 0
    assert np.allclose(res.scores64[fin], wk[fin], rtol=1e-9, atol=1e-12)
    assert not (res.rows >= n_rows).any()


def _check_gallery(m, rng, step):
    g, metric, dtype = m.g, m.metric, m.dtype
    n = len(m.rows)
    info = g.info()
    assert len(g) == n and info["rows"] == n and info["capacity"] >= n
    m.capacities.add(info["capacity"])
    assert np.array_equal(g.get_rows(np.arange(n)), m.rows)
    with pytest.raises(RuntimeError):
        g.get_rows(np.array([n]))
    if n == 0:
        return
    # queries: copies of present rows, copies of forgotten rows, random vectors (and the zero vector for DOT)
    q = [m.rows[rng.integers(0, n, 4)]]
    if m.forgotten:
        q.append(np.stack([m.forgotten[i] for i in rng.integers(0, len(m.forgotten), 3)]))
    q.append(_rand_rows(rng, 3, m.dim, metric))
    if metric == "dot":
        q.append(np.zeros((1, m.dim), np.float32))
    q = np.concatenate(q).astype(np.float32)
    Q = len(q)
    kmax = 200
    want_all = _want(metric, q, m.rows, kmax, None)
    for k in (1, 10, 200) + ((100,) if metric == "cosine" and dtype == "bf16" and step >= 4 else ()):
        res = g.search(q, k, want_scores64=True)
        _check_search(res, k, want_all, n)
        if k == 100:
            m.shadow = True           # the first k > 40 search of a bf16 COSINE gallery builds its fp16 shadow
    # a shared row mask whose last word has bits set beyond `rows`
    allowed = rng.random(n) < 0.6
    words = O.pack_row_mask(allowed)
    if n % 32:
        words[-1] |= np.uint32((0xFFFFFFFF << (n % 32)) & 0xFFFFFFFF)
    res = g.search(q, 10, row_mask=words, want_scores64=True)
    _check_search(res, 10, _want(metric, q, m.rows, 10, allowed), n)
    # two masks, one per query or none
    allowed2 = rng.random(n) < 0.3
    ids = rng.integers(-1, 2, Q).astype(np.int32)
    res = g.search(q, 10, row_mask=np.stack([O.pack_row_mask(allowed), O.pack_row_mask(allowed2)]),
                   mask_of_query=ids, want_scores64=True)
    for mid, al in ((-1, None), (0, allowed), (1, allowed2)):
        sel = ids == mid
        if sel.any():
            want = _want(metric, q[sel], m.rows, 10, al)
            assert np.array_equal(res.rows[sel], want[1]), (metric, mid)
            fin = want[1] >= 0
            assert np.allclose(res.scores64[sel][fin], want[2][fin], rtol=1e-9, atol=1e-12)
    if metric != "manhattan":
        got = g.debug_scores(q[:6])
        want, tol = raw_scores_reference(metric, dtype, q[:6], m.rows, m.shadow)
        assert got.shape == want.shape and not np.isnan(got).any()
        assert (np.abs(got - want) <= tol).all(), (metric, dtype, float(np.abs(got - want).max()))
    # the certification margin's row-norm maximum covers the 16-bit operand rows present
    op = O.round_store(m.rows, _operand_kind(metric, dtype, False)).astype(np.float64)
    assert info["max_row_norm"] >= (1 - 1e-5) * np.sqrt(np.einsum("ij,ij->i", op, op).max())


CASES = [(metric, dtype, DIMS[(i + j) % 3]) for i, metric in enumerate(METRICS) for j, dtype in enumerate(DTYPES)]


@pytest.mark.parametrize("metric,dtype,dim", CASES)
def test_mutation_sequence_against_a_numpy_model(metric, dtype, dim):
    """About a dozen seeded mutations -- appends across capacity (host and device), overwrites with host and device
    slots, a mixed overwrite + append with unsorted slots, the store's delete (get_rows(last), RAW upsert, truncate),
    truncation inside the last K3 tile, truncate(0), kernel-variant changes -- each followed by stored rows, searches
    on every path and the raw tensor-core scores against the model."""
    import torch

    from retrieval_based_object_detection_b200 import Gallery

    seed = 1000 + METRICS.index(metric) * 10 + DTYPES.index(dtype)
    rng = np.random.default_rng(seed)
    g = Gallery(dim, dtype=dtype, metric=metric, capacity=1)
    m = _Model(g, metric, dtype, dim)
    ops = ["append_host", "append_host", "append_device", "overwrite_host", "overwrite_device", "mixed", "delete",
           "truncate_tile", "variant", "append_host", "delete", "truncate_zero", "overwrite_host"]
    ops = ops[:1] + list(rng.permutation(ops[1:]))
    for step, op in enumerate(ops):
        n = len(m.rows)
        cap = g.info()["capacity"]
        if op == "append_host":
            x = _rand_rows(rng, cap - n + int(rng.integers(1, 100)), dim, metric)   # crosses the capacity: grow
            g.upsert(x)
            m.wrote(np.arange(n, n + len(x)), x)
        elif op == "append_device":
            x = _rand_rows(rng, int(rng.integers(30, 300)), dim, metric)
            g.upsert(torch.as_tensor(x, device="cuda"))
            torch.cuda.synchronize()
            m.wrote(np.arange(n, n + len(x)), x)
        elif op in ("overwrite_host", "overwrite_device") and n > 0:
            slots = rng.choice(n, size=min(n, int(rng.integers(1, 60))), replace=False)
            x = _rand_rows(rng, len(slots), dim, metric)
            m.forgotten.extend(m.rows[slots])
            if op == "overwrite_host":
                g.upsert(x, slots=slots)
            else:
                _upsert_device_slots(g, x, slots)
            m.wrote(slots, x)
        elif op == "mixed":
            old = rng.choice(n, size=min(n, 20), replace=False) if n else np.zeros(0, np.int64)
            slots = rng.permutation(np.concatenate([old, np.arange(n, n + 25)]))
            x = _rand_rows(rng, len(slots), dim, metric)
            m.forgotten.extend(m.rows[old])
            g.upsert(x, slots=slots)
            m.wrote(slots, x)
        elif op == "delete" and n > 1:
            slot, last = int(rng.integers(0, n - 1)), n - 1
            m.forgotten.append(m.rows[slot].copy())
            row = g.get_rows(np.array([last], np.int64))
            g.upsert(row, slots=np.array([slot], np.int64), raw=True)
            m.wrote([slot], row, raw=True)
            m.truncate(last)
            m.forgotten.pop()              # the moved row is still present in its new slot
        elif op == "truncate_tile" and n > 5:
            m.truncate(128 * int(rng.integers(0, (n - 6) // 128 + 1)) + 5)   # stale rows stay in the last tile
        elif op == "truncate_zero":
            m.truncate(0)
            x = _rand_rows(rng, int(rng.integers(50, 400)), dim, metric)
            g.upsert(x)
            m.wrote(np.arange(len(x)), x)
            # the reset dropped the old rows' contribution to the norm maximum
            op16 = O.round_store(m.rows, _operand_kind(metric, dtype, False)).astype(np.float64)
            want = np.sqrt(np.einsum("ij,ij->i", op16, op16).max())
            assert abs(g.info()["max_row_norm"] - want) <= 1e-5 * want
        elif op == "variant":
            g.set_option("k3_variant", int(rng.integers(0, 3)))
        _check_gallery(m, rng, step)
    assert len(m.capacities | {1024}) >= 4, sorted(m.capacities)      # 1024 and three growths at least
    g.close()


def test_forgotten_rows_stay_invisible_on_every_path():
    """A bf16 COSINE gallery large enough for the threshold pre-pass, truncated so that copies of the queries sit in
    forgotten rows, some inside the last partial K3 tile, and a 1500-row tie cluster straddles the cut."""
    from retrieval_based_object_detection_b200 import Gallery
    from test_gpu_split_search import _split_search

    n, dim, cut = 45_000, 256, 128 * 330 + 37          # 331 tiles remain: >= 320, so the pre-pass runs
    rng = np.random.default_rng(7)
    x = O.synthetic_unit_rows(n, dim, seed=70)
    q = O.synthetic_unit_rows(8, dim, seed=71)
    stale = [cut + 3, cut + 50, 128 * 331 - 1, cut + 1000, 44_000, n - 1]     # the first three in the last tile
    x[stale] = q[:6]
    tie = O.synthetic_unit_rows(1, dim, seed=72)[0]
    below = rng.choice(cut, 1100, replace=False)
    beyond = cut + rng.choice(n - cut, 400, replace=False)
    beyond = beyond[~np.isin(beyond, stale)]
    x[below], x[beyond] = tie, tie
    g = Gallery(dim, dtype="bf16", metric="cosine", capacity=n)
    g.upsert(x)
    g.truncate(cut)
    g.set_option("presample", 2)
    stored = g.get_rows(np.arange(cut))
    assert not (stored == O.l2_normalize_store(q[:6], "bf16")[0][:, None, :]).all(axis=2).any()
    for k in (10, 100):
        want_s, want_i = O.cosine_topk(q, stored, k)
        for collect in (1, 0):
            g.set_option("collect_pass", collect)
            res = g.search(q, k, want_scores64=True)
            assert np.array_equal(res.rows, want_i), (k, collect)
            assert np.allclose(res.scores64, want_s, rtol=1e-5, atol=1e-9)
            if k == 10:
                assert res.stats["presample_retries"] == 0
    survivors = np.sort(below)
    tq = tie[None, :].astype(np.float32)
    for k, collect in ((10, 1), (10, 0), (100, 1), (100, 0), (200, 1)):
        g.set_option("collect_pass", collect)
        res = g.search(tq, k, want_scores64=True)
        assert np.array_equal(res.rows[0], survivors[:k]), (k, collect)
        assert (res.rows < cut).all()
    # the split search (begin / end) on the truncated gallery, one shard (which must publish all k approximate scores)
    g.set_option("collect_pass", 1)
    for k in (10, 100):
        want_s, want_i = O.cosine_topk(q, stored, k)
        s32, ids, s64, flagged, _ = _split_search([g], [0], q, k, k)
        assert np.array_equal(ids, want_i), (k, flagged)
        np.testing.assert_allclose(s64, want_s, rtol=1e-9, atol=1e-9)
    g.close()


@pytest.mark.parametrize("device_slots", [False, True])
def test_repeated_slots_are_refused_and_change_nothing(device_slots):
    """rbod_upsert refuses a slot that appears twice: [rows + 1, rows + 1] once passed the hole check (counted as two
    fresh slots) and left slot `rows` unwritten -- zeros after a growth, or a forgotten row brought back after a
    truncate; [5, 5] raced two writers on one slot."""
    from retrieval_based_object_detection_b200 import Gallery
    from retrieval_based_object_detection_b200._native import RbodError

    rng = np.random.default_rng(5)
    dim = 256
    g = Gallery(dim, dtype="f32", metric="cosine", capacity=300)
    x = _rand_rows(rng, 300, dim, "cosine")
    g.upsert(x)
    g.truncate(200)                          # rows 200..299 are forgotten; their bytes stay in every buffer
    before = g.get_rows(np.arange(200))
    y = _rand_rows(rng, 2, dim, "cosine")

    def upsert(slots):
        if device_slots:
            _upsert_device_slots(g, y, slots)
        else:
            g.upsert(y, slots=np.asarray(slots, np.int64))

    for slots in ([201, 201], [5, 5], [200, 200]):
        with pytest.raises(RbodError):
            upsert(slots)
        assert len(g) == 200 and np.array_equal(g.get_rows(np.arange(200)), before)
        # the forgotten row at slot 200 does not come back as a hit
        res = g.search(x[200:201], 5)
        assert (res.rows < 200).all() and res.scores[0, 0] < 0.5
    upsert([201, 200])                       # distinct slots that fill [200, 201]: accepted
    assert len(g) == 202
    want = O.l2_normalize_store(y, "f32")[0]
    assert np.abs(g.get_rows(np.array([201, 200])) - want).max() <= 1e-7
    g.close()


# ------------------------------------------------------------------ the client on the device
def _client_results(c, name, queries, flt):
    """search and search_batch (with and without the filter) as comparable lists of (id, score)."""
    from qdrant_client.models import SearchRequest

    out = [[(h.id, h.score) for h in c.search(name, query_vector=v.tolist(), limit=10)] for v in queries]
    reqs = [SearchRequest(vector=v.tolist(), limit=10, filter=flt if i % 2 else None) for i, v in enumerate(queries)]
    out += [[(h.id, h.score) for h in hits] for hits in c.search_batch(name, requests=reqs)]
    return out


def _check_client_against_oracle(c, name, queries, flt, metric):
    col = c._root.get(name)
    stored = col.stored_vectors(range(len(col)))
    allowed = np.zeros(len(col), bool)
    allowed[list(col.filter_slots(flt))] = True
    got = _client_results(c, name, queries, flt)
    Q = len(queries)
    plain = _want(metric, queries, stored, 10, None)
    filtered = _want(metric, queries, stored, 10, allowed)
    for i in range(2 * Q):
        ws, wi, _ = filtered if i >= Q and (i - Q) % 2 else plain     # odd batch requests carry the filter
        r = i % Q
        hits = got[i]
        assert [col.slot_of[h[0]] for h in hits] == [int(s) for s in wi[r] if s >= 0], (i, metric)
        assert np.allclose([h[1] for h in hits], ws[r][wi[r] >= 0], rtol=1e-5, atol=1e-6)
    return got


@pytest.mark.parametrize("dtype,distance", [("bf16", "Cosine"), ("f32", "Cosine"), ("f32", "Euclid")])
def test_client_deletes_reupserts_and_reopens(store_dir, monkeypatch, dtype, distance):
    """QdrantClient on the device: 3000 points, 20 % deleted (the last slot among them), one deleted id upserted again
    with a new vector, more points -- search and search_batch equal the oracle over the stored vectors after each
    phase; a collection built from the survivors in slot order answers bit for bit the same; a reopened store (snapshot
    plus a WAL holding the deletes, then a fresh snapshot) answers bit for bit the same and scrolls the same vectors."""
    import os

    import qdrant_client as qc
    from qdrant_client.models import (Batch, Distance, FieldCondition, Filter, MatchValue, PointIdsList,
                                      VectorParams)

    monkeypatch.setenv("RBOD_GALLERY_DTYPE", dtype)
    metric = distance.lower()
    rng = np.random.default_rng(3)
    dim, n0 = 128, 3000
    c = qc.QdrantClient(host="localhost", port=6333)
    vp = VectorParams(size=dim, distance=Distance(distance))
    c.recreate_collection(collection_name="a", vectors_config=vp)
    orig = {}

    def put(name, ids, vecs):
        c.upsert(collection_name=name, points=Batch(ids=list(ids), vectors=vecs.tolist(),
                                                    payloads=[{"cls": int(i) % 5} for i in ids]))
        if name == "a":
            orig.update({int(i): v for i, v in zip(ids, vecs)})

    x = _rand_rows(rng, n0, dim, metric)
    put("a", range(n0), x)
    flt = Filter(must=[FieldCondition(key="cls", match=MatchValue(value=2))])
    col = c._root.get("a")
    queries = np.concatenate([x[rng.integers(0, n0, 4)], _rand_rows(rng, 4, dim, metric)])
    _check_client_against_oracle(c, "a", queries, flt, metric)
    c.close()                                        # snapshot now: everything below goes to the WAL

    gone = [col.ids[len(col) - 1]] + [int(i) for i in rng.choice(n0 - 1, 599, replace=False)]   # first: the last slot
    c.delete(collection_name="a", points_selector=PointIdsList(points=[int(i) for i in gone]))
    for i in gone:
        orig.pop(int(i))
    assert len(col) == n0 - 600
    queries = np.concatenate([queries, x[np.array(gone[:3])]])          # deleted vectors must not come back
    _check_client_against_oracle(c, "a", queries, flt, metric)
    back = int(gone[1])
    put("a", [back], _rand_rows(rng, 1, dim, metric))
    _check_client_against_oracle(c, "a", queries, flt, metric)
    put("a", range(n0, n0 + 700), _rand_rows(rng, 700, dim, metric))
    before = _check_client_against_oracle(c, "a", queries, flt, metric)
    scroll_before, _ = c.scroll("a", limit=100_000, with_vectors=True)

    # the survivors, upserted afresh in the first collection's slot order: the RAW moves copied stored rows exactly
    c.recreate_collection(collection_name="b", vectors_config=vp)
    put("b", list(col.ids), np.stack([orig[i] for i in col.ids]))
    assert c._root.get("b").ids == col.ids
    assert _client_results(c, "b", queries, flt) == before

    # a process that stopped here would reopen from the snapshot plus a WAL with the deletes in it
    copy = os.path.join(store_dir, "copy")
    shutil.copytree(os.path.join(store_dir, "localhost_6333"), copy)
    c_copy = qc.QdrantClient(path=copy)
    assert _client_results(c_copy, "a", queries, flt) == before
    got, _ = c_copy.scroll("a", limit=100_000, with_vectors=True)
    assert [(r.id, r.vector) for r in got] == [(r.id, r.vector) for r in scroll_before]
    qc._close_all()
    c2 = qc.QdrantClient(host="localhost", port=6333)
    assert _client_results(c2, "a", queries, flt) == before
    got, _ = c2.scroll("a", limit=100_000, with_vectors=True)
    assert [(r.id, r.vector) for r in got] == [(r.id, r.vector) for r in scroll_before]
