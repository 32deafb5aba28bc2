"""rbod_search_mmr refuses malformed requests on the host, before anything touches a device: every case returns its code
with a NULL handle (and so also here, where there is no GPU), and the message names the query and what is wrong."""
import math

import numpy as np
import pytest

from retrieval_based_object_detection_b200 import _native as N

DIM = 8


def _call(Q=2, limit=10, candidates=100, diversity=0.5, thr=None, n_masks=0, masks=None, ids=None, queries=True,
          div_null=False, outputs=True):
    lib = N.load()
    q = np.zeros((max(Q, 1), DIM), dtype=np.float32)
    div = np.broadcast_to(np.asarray(diversity, dtype=np.float64), (max(Q, 1),)).copy()
    th = None if thr is None else np.broadcast_to(np.asarray(thr, dtype=np.float32), (max(Q, 1),)).copy()
    out_s = np.empty(max(Q, 1) * max(limit, 1), dtype=np.float32)
    out_r = np.empty(max(Q, 1) * max(limit, 1), dtype=np.int64)
    ids_a = None if ids is None else np.asarray(ids, dtype=np.int32)
    masks_a = None if masks is None else np.asarray(masks, dtype=np.uint32)
    rc = lib.rbod_search_mmr(None, q.ctypes.data if queries else None, Q, limit, candidates,
                             None if div_null else div.ctypes.data, None if th is None else th.ctypes.data,
                             None if masks_a is None else masks_a.ctypes.data, n_masks,
                             None if ids_a is None else ids_a.ctypes.data, out_s.ctypes.data if outputs else None,
                             out_r.ctypes.data, None, None, None)
    return rc, lib.rbod_last_error().decode()


@pytest.mark.parametrize("kw", [
    {},
    {"Q": 0},
    {"limit": 1, "candidates": 1},
    {"limit": 1024, "candidates": 1024},
    {"diversity": [0.0, 1.0]},
    {"thr": [0.3, math.nan]},
    {"Q": 0, "div_null": True},
])
def test_well_formed_requests_reach_the_handle_check(kw):
    assert _call(**kw) == (N.RBOD_E_INVAL, "rbod_search_mmr: NULL handle")


@pytest.mark.parametrize("kw,msg", [
    ({"limit": 0}, "limit = 0 < 1"),
    ({"limit": 10, "candidates": 9}, "candidates = 9 < limit = 10"),
    ({"diversity": [0.5, math.nan]}, "query 1: diversity nan is not in [0, 1]"),
    ({"diversity": [-0.1, 0.5]}, "query 0: diversity -0.1 is not in [0, 1]"),
    ({"diversity": [0.5, 1.5]}, "query 1: diversity 1.5 is not in [0, 1]"),
    ({"div_null": True}, "diversity is NULL"),
    ({"queries": False}, "NULL queries or outputs"),
    ({"outputs": False}, "NULL queries or outputs"),
    ({"Q": -1}, "Q = -1 out of range"),
    ({"n_masks": -1}, "-1 masks, row_masks NULL"),
    ({"n_masks": 1}, "1 masks, row_masks NULL"),
    ({"n_masks": 2, "masks": np.zeros((2, 1)), "ids": [0, 2]}, "query 1: mask_of_query = 2 is outside [-1, 2)"),
    ({"n_masks": 2, "masks": np.zeros((2, 1)), "ids": [-2, 0]}, "query 0: mask_of_query = -2 is outside [-1, 2)"),
    ({"ids": [-1, 0]}, "query 1: mask_of_query = 0 is outside [-1, 0)"),
])
def test_malformed_requests(kw, msg):
    rc, text = _call(**kw)
    assert rc == N.RBOD_E_INVAL and text == "rbod_search_mmr: " + msg, text


def test_candidates_beyond_1024_are_unsupported():
    assert _call(candidates=1025) == (N.RBOD_E_UNSUPPORTED, "rbod_search_mmr: candidates = 1025 > 1024")
    # malformed requests are reported first
    assert _call(candidates=1025, diversity=2.0)[0] == N.RBOD_E_INVAL
    # valid masks pass on to the handle check
    assert _call(n_masks=2, masks=np.zeros((2, 1)), ids=[1, -1])[1] == "rbod_search_mmr: NULL handle"
