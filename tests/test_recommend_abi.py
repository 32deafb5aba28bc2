"""rbod_recommend refuses malformed requests on the host, before anything touches a device: every case returns its code
with a NULL handle (and so also here, where there is no GPU), and the message names what is wrong."""
import ctypes

import numpy as np
import pytest

from retrieval_based_object_detection_b200 import _native as N

DIM = 8


def _call(offsets, signs, k=10, R=None, n_masks=0, masks=None, ids=None, examples=True):
    lib = N.load()
    off = np.asarray(offsets, dtype=np.int64)
    sg = np.asarray(signs, dtype=np.int8)
    R = len(off) - 1 if R is None else R
    E = len(sg)
    ex = np.zeros((max(E, 1), DIM), dtype=np.float32)
    out_s = np.empty(max(R, 1) * k, dtype=np.float32)
    out_r = np.empty(max(R, 1) * k, dtype=np.int64)
    ids_a = None if ids is None else np.asarray(ids, dtype=np.int32)
    masks_a = None if masks is None else np.asarray(masks, dtype=np.uint32)
    rc = lib.rbod_recommend(None, ex.ctypes.data if examples else None, E, sg.ctypes.data, off.ctypes.data, R, k,
                            None if masks_a is None else masks_a.ctypes.data, n_masks,
                            None if ids_a is None else ids_a.ctypes.data, out_s.ctypes.data, out_r.ctypes.data, None,
                            None, None)
    return rc, lib.rbod_last_error().decode()


def test_a_well_formed_request_reaches_the_handle_check():
    assert _call([0, 2, 3], [1, -1, 1]) == (N.RBOD_E_INVAL, "rbod_recommend: NULL handle")
    assert _call([0], [], R=0)[1] == "rbod_recommend: NULL handle"


@pytest.mark.parametrize("offsets,signs,what", [
    ([0, 0, 2], [1, 1], "has 0 examples"),                       # an empty request
    ([0, 33], [1] * 33, "has 33 examples"),                      # more than 32 examples
    ([0, 3, 2, 4], [1] * 4, "has -1 examples"),                  # offsets not monotone
    ([1, 3], [1, 1, 1], "from 0 to n_examples"),                 # not starting at 0
    ([0, 2], [1, 1, 1], "from 0 to n_examples"),                 # not ending at n_examples
    ([0, 2, 3], [1, 0, -1], "example_sign[1] = 0"),              # a sign other than +1 / -1
    ([0, 2, 3], [1, -1, 2], "example_sign[2] = 2"),
])
def test_malformed_requests(offsets, signs, what):
    rc, msg = _call(offsets, signs)
    assert rc == N.RBOD_E_INVAL and what in msg, msg


def test_malformed_masks_and_k():
    masks = np.zeros((2, 1), dtype=np.uint32)
    assert _call([0, 1, 2], [1, 1], n_masks=2, masks=masks, ids=[0, 2])[1].endswith("mask_of_request[1] = 2 is outside [-1, 2)")
    assert _call([0, 1, 2], [1, 1], n_masks=2, masks=masks, ids=[-2, 0])[1].endswith("mask_of_request[0] = -2 is outside [-1, 2)")
    assert _call([0, 1, 2], [1, 1], n_masks=0, ids=[0, -1])[1].endswith("mask_of_request[0] = 0 is outside [-1, 0)")
    assert _call([0, 1], [1], n_masks=-1) == (N.RBOD_E_INVAL, "rbod_recommend: -1 masks, row_masks NULL")
    assert _call([0, 1], [1], n_masks=1) == (N.RBOD_E_INVAL, "rbod_recommend: 1 masks, row_masks NULL")
    assert _call([0, 1], [1], k=0) == (N.RBOD_E_INVAL, "rbod_recommend: k = 0 < 1")
    assert _call([0, 1], [1], examples=False)[1] == "rbod_recommend: NULL examples, signs, offsets or outputs"
    # masks and ids that are valid pass on to the handle check; k beyond the sweep's lists is unsupported
    assert _call([0, 1, 2], [1, 1], n_masks=2, masks=masks, ids=[1, -1])[1] == "rbod_recommend: NULL handle"
    assert _call([0, 1], [1], k=1025) == (N.RBOD_E_UNSUPPORTED, "rbod_recommend: k=1025 > 1024")
    assert _call([0, 1], [1], k=1024)[1] == "rbod_recommend: NULL handle"
