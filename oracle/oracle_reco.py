"""fp64 numpy oracle of recommendation by the best_score rule (include/rbod.h, rbod_recommend).

For an example e and a stored row g the key is the exact search ordering key (COSINE dot/(|e||g|), DOT dot, EUCLID
-sum (e-g)^2, MANHATTAN -sum |e-g|) in float64 from the float32 example and the stored row.  Per request:
bp / bn = the largest key over its positives / negatives (-inf when there are none), sim(x) = x (-sqrt(-x) for
EUCLID), s(y) = 0.5 * (y / (1 + |y|) + 1), and the score is s(sim(bp)) if bp > bn, else -s(sim(bn)).  This is the
best_score rule of Qdrant >= 1.7 (merge_similarities / scaled_fast_sigmoid) as read from its source; it has not been
compared with a live Qdrant.

Identical stored rows get bit-identical keys here (the keys are computed once per distinct row), so a test that
plants a tie cluster sees the ties the device sees.
"""
from __future__ import annotations

import numpy as np

from . import oracle_np as O


def example_keys(examples, stored, metric: str) -> np.ndarray:
    """[E, n] float64 keys of every (example, stored row) pair."""
    e = np.atleast_2d(np.asarray(examples, dtype=np.float32)).astype(np.float64)
    g32 = np.atleast_2d(np.asarray(stored, dtype=np.float32))
    if len(g32) == 0:
        return np.zeros((len(e), 0))
    uniq, inv = np.unique(g32, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    g = uniq.astype(np.float64)
    if metric in ("cosine", "dot"):
        dots = e @ g.T
        if metric == "dot":
            keys = dots
        else:
            den = np.sqrt(np.einsum("ij,ij->i", e, e))[:, None] * np.sqrt(np.einsum("ij,ij->i", g, g))[None, :]
            with np.errstate(divide="ignore", invalid="ignore"):
                keys = np.where(den > 0.0, dots / den, 0.0)
    elif metric in ("euclid", "manhattan"):
        keys = np.empty((len(e), len(g)))
        for i in range(len(e)):
            d = g - e[i][None, :]
            keys[i] = -(d * d).sum(axis=1) if metric == "euclid" else -np.abs(d).sum(axis=1)
    else:
        raise ValueError(metric)
    return keys[:, inv]


def _s(y):
    return 0.5 * (y / (1.0 + np.abs(y)) + 1.0)


def best_score(keys, signs, offsets, metric: str) -> np.ndarray:
    """[E, n] example keys -> [R, n] best_score scores of the requests given by ``offsets`` [R + 1] and ``signs`` [E]."""
    keys = np.asarray(keys, dtype=np.float64)
    signs = np.asarray(signs)
    offsets = np.asarray(offsets, dtype=np.int64)
    sim = (lambda x: -np.sqrt(-x)) if metric == "euclid" else (lambda x: x)
    out = np.empty((len(offsets) - 1, keys.shape[1]))
    for r in range(len(offsets) - 1):
        kk, sg = keys[offsets[r]:offsets[r + 1]], signs[offsets[r]:offsets[r + 1]]
        bp = kk[sg > 0].max(axis=0) if (sg > 0).any() else np.full(keys.shape[1], -np.inf)
        bn = kk[sg < 0].max(axis=0) if (sg < 0).any() else np.full(keys.shape[1], -np.inf)
        with np.errstate(invalid="ignore"):
            pos = _s(sim(bp))
            neg = -_s(sim(bn))
        out[r] = np.where(bp > bn, pos, neg)
    return out


def recommend_topk(examples, signs, offsets, stored, k: int, metric: str, allowed=None):
    """Exact best_score top-k per request, ordered by (score desc, row asc), padded with (-inf, -1).
    ``allowed``: None, or one bool[n] row mask (or None) per request.  -> (scores f64 [R, k], rows i64 [R, k])."""
    sc = best_score(example_keys(examples, stored, metric), signs, offsets, metric)
    R = sc.shape[0]
    out_s = np.full((R, k), -np.inf)
    out_i = np.full((R, k), -1, dtype=np.int64)
    for r in range(R):
        m = None if allowed is None else allowed[r]
        out_s[r], out_i[r] = (x[0] for x in O.topk_from_scores(sc[r:r + 1], k, row_mask=m))
    return out_s, out_i


def agrees(got_rows, got_keys, scores, want_keys, want_rows, rtol: float = 1e-12) -> bool:
    """Whether one request's device top-k (``got_rows`` / ``got_keys``) agrees with the oracle's (``want_keys`` /
    ``want_rows``, from ``scores`` [n], the oracle's scores of every row).  The rows must be distinct, ordered by
    (key desc, row asc), padded exactly where the oracle pads, and the oracle's score of the row at every rank must be
    the oracle's score of that rank within ``rtol``; the keys themselves within ``rtol`` too.  So ids can differ from the
    oracle's only among rows whose scores lie within ``rtol`` of each other, which two fp64 sums taken in different
    orders cannot order reliably (a stored row given as its own example scores s(1) give or take an ulp)."""
    got_rows, got_keys = np.asarray(got_rows), np.asarray(got_keys, dtype=np.float64)
    valid = np.asarray(want_rows) >= 0
    if not np.array_equal(got_rows >= 0, valid) or not np.all(np.isneginf(got_keys[~valid])):
        return False
    g, gk, wk = got_rows[valid], got_keys[valid], np.asarray(want_keys)[valid]
    if len(np.unique(g)) != len(g) or np.any((gk[1:] > gk[:-1]) | ((gk[1:] == gk[:-1]) & (g[1:] < g[:-1]))):
        return False
    return bool(np.allclose(scores[g], wk, rtol=rtol, atol=0) and np.allclose(gk, wk, rtol=rtol, atol=0))
