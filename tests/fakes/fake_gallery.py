"""TEST DOUBLE for ``retrieval_based_object_detection_b200.gallery.Gallery`` -- test infrastructure only.

It answers the Gallery interface with the CPU oracle so the HOST side of the drop-in (ids, payload filters,
scroll paging, staging, persistence, the call sequences of the reference's scripts) can be exercised in the
``-m "not gpu"`` suite, where no B200 exists.  The product never imports this module and has no CPU path; the
``-m gpu`` tests run the same scenarios against the real library.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

from oracle import oracle_np as O


class FakeGallery:
    def __init__(self, dim, dtype="f32", metric="cosine", capacity=0, device=0):
        self.dim, self.dtype, self.metric, self.device = int(dim), dtype, metric, device
        self._rows = np.zeros((0, self.dim), dtype=np.float32)
        self.calls = []

    def __len__(self):
        return len(self._rows)

    count = property(__len__)

    def close(self):
        pass

    def truncate(self, rows):
        assert 0 <= rows <= len(self._rows)
        self._rows = self._rows[:rows].copy()

    def set_option(self, key, value):
        pass

    def upsert(self, rows, slots=None, return_norms=False, raw=False, stream=None):
        rows = np.ascontiguousarray(rows, dtype=np.float32).reshape(-1, self.dim)
        self.calls.append(("upsert", len(rows)))
        if raw or self.metric != "cosine":
            stored, norms = O.round_store(rows, self.dtype), np.linalg.norm(rows.astype(np.float64), axis=1)
        else:
            stored, norms = O.l2_normalize_store(rows, self.dtype)
        if slots is None:
            slots = np.arange(len(self._rows), len(self._rows) + len(rows))
        slots = np.asarray(slots, dtype=np.int64)
        # refused like rbod_upsert does: repeated slots, negative slots, slots that leave holes
        if len(np.unique(slots)) != len(slots):
            raise RuntimeError("rbod_upsert: slot appears more than once")
        if len(slots) and slots.min() < 0:
            raise RuntimeError("rbod_upsert: negative slot")
        if len(slots) and slots.max() + 1 > len(self._rows) + int((slots >= len(self._rows)).sum()):
            raise RuntimeError("rbod_upsert: slots would leave holes")
        new_n = max(len(self._rows), int(slots.max()) + 1 if len(slots) else 0)
        if new_n > len(self._rows):
            grown = np.zeros((new_n, self.dim), dtype=np.float32)
            grown[: len(self._rows)] = self._rows
            self._rows = grown
        self._rows[slots] = stored
        return norms.astype(np.float32) if return_norms else None

    def get_rows(self, rows):
        rows = np.asarray(rows, dtype=np.int64)
        if len(rows) and (rows.min() < 0 or rows.max() >= len(self._rows)):
            raise RuntimeError("row index outside the gallery")
        return self._rows[rows].copy()

    def segment_mean(self, offsets, row_idx=None):
        offsets = np.asarray(offsets, dtype=np.int64)
        row_idx = np.arange(offsets[-1]) if row_idx is None else np.asarray(row_idx, dtype=np.int64)
        self.calls.append(("segment_mean", len(offsets) - 1))
        return O.segment_mean_renorm(self._rows, row_idx, offsets, normalize=self.metric == "cosine")

    def segment_delegates(self, kind, offsets, row_idx=None, alpha=2.0):
        fn = {"average": O.compute_average, "centroid": O.compute_centroid, "medoid": O.compute_medoid,
              "weighted": lambda v: O.compute_weighted_average(v, alpha)}[kind]
        offsets = np.asarray(offsets, dtype=np.int64)
        row_idx = np.arange(offsets[-1]) if row_idx is None else np.asarray(row_idx, dtype=np.int64)
        return (O.segment_mean_renorm(self._rows, row_idx, offsets, average_fn=fn, normalize=self.metric == "cosine"),
                np.full(len(offsets) - 1, -1))

    def search(self, queries, k, row_mask=None, want_scores64=False, out=None, stream=None):
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        self.calls.append(("search", len(q), k))
        allowed = None if row_mask is None else O.unpack_row_mask(np.asarray(row_mask), len(self._rows))
        if len(self._rows) == 0:
            s = np.full((len(q), k), -np.inf)
            i = np.full((len(q), k), -1, dtype=np.int64)
        elif self.metric in ("euclid", "manhattan"):
            d, i, keys = O.distance_topk(q, self._rows, k, self.metric, row_mask=allowed)
            return SimpleNamespace(scores=d.astype(np.float32), rows=i, scores64=keys, stats={})
        else:
            s, i = O.cosine_topk(q, self._rows, k, row_mask=allowed)
        return SimpleNamespace(scores=s.astype(np.float32), rows=i, scores64=s, stats={})


def install():
    """Routes every Gallery the host layer creates to the double (call before touching a collection)."""
    import retrieval_based_object_detection_b200 as pkg
    import retrieval_based_object_detection_b200.gallery as gallery

    gallery.Gallery = FakeGallery
    pkg.Gallery = FakeGallery
