"""rbod_discover refuses malformed requests on the host, before anything touches a device: every case returns its code
with a NULL handle (and so also here, where there is no GPU), and the message names the request and what is wrong."""
import numpy as np
import pytest

from retrieval_based_object_detection_b200 import _native as N

DIM = 8


def _call(offsets, roles, k=10, R=None, n_masks=0, masks=None, ids=None, examples=True):
    lib = N.load()
    off = np.asarray(offsets, dtype=np.int64)
    rl = np.asarray(roles, dtype=np.int8)
    R = len(off) - 1 if R is None else R
    E = len(rl)
    ex = np.zeros((max(E, 1), DIM), dtype=np.float32)
    out_s = np.empty(max(R, 1) * k, dtype=np.float32)
    out_r = np.empty(max(R, 1) * k, dtype=np.int64)
    ids_a = None if ids is None else np.asarray(ids, dtype=np.int32)
    masks_a = None if masks is None else np.asarray(masks, dtype=np.uint32)
    rc = lib.rbod_discover(None, ex.ctypes.data if examples else None, E, rl.ctypes.data, off.ctypes.data, R, k,
                           None if masks_a is None else masks_a.ctypes.data, n_masks,
                           None if ids_a is None else ids_a.ctypes.data, out_s.ctypes.data, out_r.ctypes.data, None,
                           None, None)
    return rc, lib.rbod_last_error().decode()


@pytest.mark.parametrize("offsets,roles", [
    ([0, 5, 7], [0, 1, -1, 1, -1, 1, -1]),      # a discovery request and a context request
    ([0, 1], [0]),                              # a target alone
    ([0, 31], [0] + [1, -1] * 15),              # a target and 15 pairs
    ([0, 32], [1, -1] * 16),                    # 16 pairs without a target
    ([0], []),                                  # no request
])
def test_well_formed_requests_reach_the_handle_check(offsets, roles):
    assert _call(offsets, roles) == (N.RBOD_E_INVAL, "rbod_discover: NULL handle")


@pytest.mark.parametrize("offsets,roles,what", [
    ([0, 0, 2], [1, -1], "request 0 has 0 examples"),                        # an empty request
    ([0, 33], [0] + [1, -1] * 16, "request 0 has 33 examples"),             # more than 32 examples
    ([0, 3, 2, 4], [1, -1, 1, -1], "request 1 has -1 examples"),            # offsets not monotone
    ([1, 3], [0, 1, -1], "from 0 to n_examples"),                           # not starting at 0
    ([0, 2], [0, 1, -1], "from 0 to n_examples"),                           # not ending at n_examples
    ([0, 3], [0, 2, -1], "example_role[1] = 2 is not 0, +1 or -1"),         # a role outside {0, +-1}
    ([0, 1, 4], [0, 1, -1, -2], "example_role[3] = -2 is not 0, +1 or -1"),
    ([0, 3], [1, -1, 0], "request 0: a target at example 2"),               # a target that is not first
    ([0, 1, 5], [0, 0, 0, 1, -1], "request 1: a second target at example 2"),   # a second target
    ([0, 2], [0, 1], "request 0: positive example 1 is not followed by a negative"),
    ([0, 3], [1, 1, -1], "request 0: positive example 0 is not followed by a negative"),
    ([0, 2], [0, -1], "request 0: negative example 1 is not preceded by a positive"),
    ([0, 1, 2], [0, -1], "request 1: negative example 1 is not preceded by a positive"),
    ([0, 3], [1, -1, -1], "request 0: negative example 2 is not preceded by a positive"),
    ([0, 1], [1], "request 0: positive example 0 is not followed by a negative"),   # neither a target nor a pair
])
def test_malformed_requests(offsets, roles, what):
    rc, msg = _call(offsets, roles)
    assert rc == N.RBOD_E_INVAL and what in msg, msg
    assert msg.startswith("rbod_discover: ")


def test_malformed_masks_and_k():
    masks = np.zeros((2, 1), dtype=np.uint32)
    assert _call([0, 1, 3], [0, 1, -1], n_masks=2, masks=masks, ids=[0, 2])[1].endswith(
        "mask_of_request[1] = 2 is outside [-1, 2)")
    assert _call([0, 1, 2], [0, 0], n_masks=2, masks=masks, ids=[-2, 0])[1].endswith(
        "mask_of_request[0] = -2 is outside [-1, 2)")
    assert _call([0, 1, 2], [0, 0], n_masks=0, ids=[0, -1])[1].endswith("mask_of_request[0] = 0 is outside [-1, 0)")
    assert _call([0, 1], [0], n_masks=-1) == (N.RBOD_E_INVAL, "rbod_discover: -1 masks, row_masks NULL")
    assert _call([0, 1], [0], n_masks=1) == (N.RBOD_E_INVAL, "rbod_discover: 1 masks, row_masks NULL")
    assert _call([0, 1], [0], k=0) == (N.RBOD_E_INVAL, "rbod_discover: k = 0 < 1")
    assert _call([0, 1], [0], examples=False)[1] == "rbod_discover: NULL examples, roles, offsets or outputs"
    # masks and ids that are valid pass on to the handle check; k beyond the sweep's lists is unsupported
    assert _call([0, 1, 3], [0, 1, -1], n_masks=2, masks=masks, ids=[1, -1])[1] == "rbod_discover: NULL handle"
    assert _call([0, 1], [0], k=1025) == (N.RBOD_E_UNSUPPORTED, "rbod_discover: k=1025 > 1024")
    assert _call([0, 1], [0], k=1024)[1] == "rbod_discover: NULL handle"
