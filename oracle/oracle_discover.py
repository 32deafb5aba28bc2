"""fp64 numpy oracle of discovery and context search (include/rbod.h, rbod_discover).

Keys are oracle_reco's ``example_keys`` (identical stored rows get bit-identical keys), sim and s are best_score's:
sim(x) = x (-sqrt(-x) for EUCLID), s(y) = 0.5 (f(y) + 1) with f(y) = y / (1 + |y|), and MARGIN = 2^-23 (f32 epsilon).
For a pair (p, n) and a row g with P = key(p, g), N = key(n, g):
  rank_pair = +1 if P > N else -1 (a tie counts -1);  loss_pair = f(min(sim(P) - sim(N) - MARGIN, 0)).
A request with a target t (discovery) scores sum(rank_pair) + s(sim(key(t, g))); one without (context) scores the sum of
its loss_pair in pair order, 0 for every row on the positive side of every pair.  This is the rule of Qdrant >= 1.7
(DiscoveryQuery::score_by, ContextPair::loss_by) as read from its source; it has not been compared with a live Qdrant.
Device answers are compared with oracle_reco's ``agrees``.
"""
from __future__ import annotations

import numpy as np

from . import oracle_np as O
from .oracle_reco import example_keys

MARGIN = 2.0 ** -23   # f32 epsilon: a context pair's loss is 0 only when sim(P) - sim(N) reaches it


def _f(y):
    return y / (1.0 + np.abs(y))


def discover_score(keys, roles, offsets, metric: str) -> np.ndarray:
    """[E, n] example keys -> [R, n] discovery / context scores of the requests given by ``offsets`` [R + 1] and
    ``roles`` [E] (0 = the target, first; then (+1, -1) pairs)."""
    keys = np.asarray(keys, dtype=np.float64)
    roles = np.asarray(roles)
    offsets = np.asarray(offsets, dtype=np.int64)
    sim = (lambda x: -np.sqrt(-x)) if metric == "euclid" else (lambda x: x)
    out = np.empty((len(offsets) - 1, keys.shape[1]))
    for r in range(len(offsets) - 1):
        kk, rl = keys[offsets[r]:offsets[r + 1]], roles[offsets[r]:offsets[r + 1]]
        has_target = rl[0] == 0
        rank = np.zeros(keys.shape[1], dtype=np.int64)
        loss = np.zeros(keys.shape[1])
        for P, N in zip(kk[1 if has_target else 0::2], kk[2 if has_target else 1::2]):
            rank += np.where(P > N, 1, -1)
            with np.errstate(invalid="ignore"):
                loss = loss + _f(np.minimum(sim(P) - sim(N) - MARGIN, 0.0))
        out[r] = rank + 0.5 * (_f(sim(kk[0])) + 1.0) if has_target else loss
    return out


def discover_topk(examples, roles, offsets, stored, k: int, metric: str, allowed=None):
    """Exact discovery / context top-k per request, ordered by (score desc, row asc), padded with (-inf, -1).
    ``allowed``: None, or one bool[n] row mask (or None) per request.  -> (scores f64 [R, k], rows i64 [R, k])."""
    sc = discover_score(example_keys(examples, stored, metric), roles, offsets, metric)
    R = sc.shape[0]
    out_s = np.full((R, k), -np.inf)
    out_i = np.full((R, k), -1, dtype=np.int64)
    for r in range(R):
        m = None if allowed is None else allowed[r]
        out_s[r], out_i[r] = (x[0] for x in O.topk_from_scores(sc[r:r + 1], k, row_mask=m))
    return out_s, out_i
