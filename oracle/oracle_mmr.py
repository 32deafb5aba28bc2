"""fp64 numpy oracle of maximal marginal relevance (include/rbod.h, rbod_search_mmr).

For a query q the candidates c_0 .. c_{L-1} are the exact top-L by the search key (oracle_np's ``topk_from_scores``,
ordered by key desc, row asc), keeping those whose fp32 search score passes the threshold (>=, or <= for the distances
of EUCLID / MANHATTAN).  With sim(y) = y (-sqrt(-y) for EUCLID), rel(c) = sim(key(q, c)) and lambda = 1 - diversity, the
first pick is c_0 and every later pick maximises
    mmr(c) = lambda * rel(c) - diversity * max over picked s of sim(key(s, c))
over the unpicked candidates, exact ties to the smaller candidate rank.  Results come in selection order.  Keys are
oracle_reco's ``example_keys``, so identical stored rows get bit-identical keys.  Qdrant >= 1.15 documents the same kind
of rule; this one has not been checked against a live Qdrant or its source.
"""
from __future__ import annotations

import numpy as np

from . import oracle_np as O
from .oracle_reco import example_keys


def sim(keys, metric: str):
    keys = np.asarray(keys, dtype=np.float64)
    return -np.sqrt(-keys) if metric == "euclid" else keys


def user_scores(keys, metric: str) -> np.ndarray:
    """fp64 search keys -> the fp32 scores a search reports (the distance for EUCLID / MANHATTAN)."""
    keys = np.asarray(keys, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        if metric == "euclid":
            return np.sqrt(-keys).astype(np.float32)
        if metric == "manhattan":
            return (-keys).astype(np.float32)
    return keys.astype(np.float32)


def candidates(query, stored, L: int, metric: str, allowed=None, score_threshold=None, qkeys=None):
    """-> (rows i64 [n], keys f64 [n]): the exact top-L of ``query`` that take part (n <= L).  ``qkeys``: the query's
    [n_rows] keys, when they were computed for several queries at once."""
    qk = (example_keys(np.asarray(query, np.float32).reshape(1, -1), stored, metric) if qkeys is None
          else np.asarray(qkeys, np.float64).reshape(1, -1))
    ks, ki = O.topk_from_scores(qk, L, row_mask=allowed)
    ok = ki[0] >= 0
    if score_threshold is not None and not np.isnan(score_threshold):
        sc = user_scores(ks[0], metric)
        with np.errstate(invalid="ignore"):
            ok &= (sc <= np.float32(score_threshold)) if metric in ("euclid", "manhattan") else (sc >= np.float32(score_threshold))
    n = int(np.argmin(ok)) if not ok.all() else len(ok)   # a prefix: the score is monotone in the key
    return ki[0][:n], ks[0][:n]


def mmr_step_values(rel, pair_sim, picked, diversity: float) -> np.ndarray:
    """mmr of every candidate given the picks so far (``picked``: candidate ranks), -inf for picked ones."""
    lam = 1.0 - diversity
    ms = pair_sim[list(picked)].max(axis=0)
    v = lam * rel - diversity * ms
    v[list(picked)] = -np.inf
    return v


def prepare(query, stored, L: int, metric: str, allowed=None, score_threshold=None, qkeys=None):
    """What a query's selection needs whatever its limit and diversity: (candidate rows, their keys, rel, pair_sim with
    pair_sim[s, c] = sim(key(s, c)) over the candidates)."""
    stored = np.asarray(stored, np.float32)
    rows, keys = candidates(query, stored, L, metric, allowed, score_threshold, qkeys)
    pair_sim = sim(example_keys(stored[rows], stored[rows], metric), metric) if len(rows) else np.zeros((0, 0))
    return rows, keys, sim(keys, metric), pair_sim


def mmr_select(query, stored, limit: int, L: int, diversity: float, metric: str, allowed=None, score_threshold=None,
               prepared=None):
    """-> (rows i64 [limit], keys f64 [limit]) in selection order, padded with (-1, -inf).  ``prepared``: the query's
    ``prepare`` result, when several selections share it."""
    rows, keys, rel, pair_sim = prepared or prepare(query, stored, L, metric, allowed, score_threshold)
    out_r = np.full(limit, -1, dtype=np.int64)
    out_k = np.full(limit, -np.inf)
    n = len(rows)
    if n == 0:
        return out_r, out_k
    picked = [0]
    while len(picked) < min(limit, n):
        v = mmr_step_values(rel, pair_sim, picked, diversity)
        picked.append(int(np.argmax(v)))   # argmax takes the first of equal values: the smaller rank
    out_r[:len(picked)] = rows[picked]
    out_k[:len(picked)] = keys[picked]
    return out_r, out_k


def mmr_agrees(got_rows, query, stored, limit: int, L: int, diversity: float, metric: str, allowed=None,
               score_threshold=None, prepared=None) -> bool:
    """Replay of one query's device answer ``got_rows`` (selection order, -1 padded) against the oracle:
    * every picked row is one of the exact top-L candidates (a row outside them is allowed only if its key ties the
      L-th candidate's within the tolerance below, where two fp64 sums taken in different orders cannot order rows);
    * at every step the device's pick is unpicked and reaches the oracle's best mmr given the device's earlier picks,
      within 1e-12 (1 + max |rel| + max |sim|);
    * padding sits where the oracle's does (min(limit, candidates that take part) picks)."""
    stored = np.asarray(stored, np.float32)
    got_rows = np.asarray(got_rows, dtype=np.int64)
    rows, keys, rel, pair_sim = prepared or prepare(query, stored, L, metric, allowed, score_threshold)
    n = len(rows)
    picks = min(limit, n)
    if not (np.all(got_rows[:picks] >= 0) and np.all(got_rows[picks:] == -1)):
        return False
    if picks == 0:
        return True
    got = got_rows[:picks]
    if len(np.unique(got)) != picks:
        return False
    # rows at the boundary of the top L that tie with the L-th key within the tolerance may stand in for it
    extra = np.setdiff1d(got, rows)
    if len(extra):
        qk = example_keys(np.asarray(query, np.float32).reshape(1, -1), stored, metric)[0]
        tol_k = 1e-12 * (1.0 + np.abs(keys).max())
        if np.any(qk[extra] < keys[-1] - tol_k):
            return False
        rows = np.concatenate([rows, extra])
        keys = np.concatenate([keys, qk[extra]])
        rel = sim(keys, metric)
        pair_sim = sim(example_keys(stored[rows], stored[rows], metric), metric)
    tol = 1e-12 * (1.0 + np.abs(rel).max() + np.abs(pair_sim).max())
    rank = {int(r): i for i, r in enumerate(rows)}
    if rank[int(got[0])] != 0 and not rel[rank[int(got[0])]] >= rel[0] - tol:
        return False
    picked = [rank[int(got[0])]]
    for r in got[1:]:
        j = rank[int(r)]
        if j in picked:
            return False
        v = mmr_step_values(rel, pair_sim, picked, diversity)
        if v[j] < v.max() - tol:
            return False
        picked.append(j)
    return True
