"""Host side of a collection: point ids, payloads, filters, persistence, upsert staging.

This is the part of the (third-party) Qdrant server the reference scripts rely on that is NOT
arithmetic: everything here is bookkeeping in Python; every vector operation goes to a
``Gallery`` (librbod.so).  Behaviours reproduced, with the reference call sites that need them:

* upsert-overwrites-by-id with deterministic md5 ids   31_…py:42-43,177-179; 32_…py:29-31,41-42
* ids are unsigned ints or UUID strings, returned canonical (hyphenated)
* scroll pages ordered by id (ints first, then UUIDs), ``limit`` default 10, ``next_page_offset``
                                                       32_…py:78-82,123-131; 33_…py:96-106,139-145
* ``Filter(must=[FieldCondition(key, match=MatchValue(value))])`` = AND of payload equalities;
  a ``None`` payload value never matches                 32_…py:125-129; 33_…py:98-103,117-137
* state survives the process (the scripts are separate processes talking to one server):
  ``meta.json`` + a versioned snapshot (``snap-<N>/points.json`` + ``snap-<N>/vectors.npy``, made current by
  an atomic rename of the ``CURRENT`` pointer file) + an append-only ``wal.jsonl`` replayed in log order.

Single-point upserts (31_…py:179 sends one RPC per image) are appended to the WAL and kept in a
host staging dict; they reach the GPU in one batched K1 launch on the first read that needs
vectors, so read-your-writes holds without a kernel launch per point.
"""
from __future__ import annotations

import base64
import copy
import json
import os
import shutil
import uuid
from typing import Any, Dict, Iterable, List, Optional, Sequence, Set

import numpy as np

FORMAT_VERSION = 1
_FLUSH_THRESHOLD = 65536  # staged rows that force a device flush
MAX_RECOMMEND_EXAMPLES = 32   # examples per recommendation / discovery request (rbod_recommend, rbod_discover)
MAX_RECOMMEND_FETCH = 1024    # rows such a request fetches: limit + offset + its example ids


class CollectionNotFound(Exception):
    """Raised for operations on a collection that does not exist (the server's 404)."""

    def __init__(self, name: str):
        super().__init__(f"Not found: Collection `{name}` doesn't exist!")
        self.status_code = 404
        self.collection = name


def canonical_id(pid) -> Any:
    """Qdrant point id rules: unsigned 64-bit int, or a UUID given in any textual form."""
    if isinstance(pid, bool):
        raise ValueError(f"invalid point id {pid!r}")
    if isinstance(pid, (int, np.integer)):
        v = int(pid)
        if v < 0 or v >= 1 << 64:
            raise ValueError(f"point id {v} is not an unsigned 64-bit integer")
        return v
    if isinstance(pid, uuid.UUID):
        return str(pid)
    if isinstance(pid, str):
        try:
            return str(uuid.UUID(pid))
        except ValueError as exc:
            raise ValueError(f"point id {pid!r} is neither an unsigned integer nor a UUID") from exc
    raise ValueError(f"unsupported point id type {type(pid).__name__}")


def id_sort_key(pid):
    return (0, pid) if isinstance(pid, int) else (1, uuid.UUID(pid).int)


def _vkey(value):
    """Index key that keeps True / 1 / 1.0 / "1" apart (python would merge the first three)."""
    return (type(value).__name__, value)


def _indexable(value) -> bool:
    return isinstance(value, (str, bool, int, float)) and value is not None


class Collection:
    """One collection: host metadata + (lazily) a device gallery."""

    def __init__(self, directory: Optional[str], name: str, dim: int, distance: str, dtype: str = "f32",
                 device: int = 0):
        self.directory = directory  # None = in-memory only
        self.name = name
        self.dim = int(dim)
        self.distance = distance
        self.dtype = dtype
        self.device = device
        self.ids: List[Any] = []
        self.slot_of: Dict[Any, int] = {}
        self.payloads: List[dict] = []
        self.index: Dict[str, Dict[Any, Set[int]]] = {}
        self.list_keys: Set[str] = set()    # payload keys that ever held a list: matched per element, never by column
        self.pending: Dict[int, np.ndarray] = {}
        self.snapshot_vectors: Optional[np.ndarray] = None  # stored rows loaded from disk, not yet on device
        self.snap_src: Optional[np.ndarray] = None          # slot -> row of snapshot_vectors (-1: vector is staged)
        self._snap_no = 0                                   # number of the current snapshot directory
        self.gallery = None
        self._order: Optional[List[int]] = None
        self._columns: Dict[str, Any] = {}     # key -> (int32 codes per slot, {value key -> code}); rebuilt lazily
        self._columns_n = -1
        self._dirty = False
        self._wal = None

    # ------------------------------------------------------------------ persistence
    @staticmethod
    def meta_path(directory: str) -> str:
        return os.path.join(directory, "meta.json")

    @classmethod
    def create(cls, directory: Optional[str], name: str, dim: int, distance: str, dtype: str, device: int):
        col = cls(directory, name, dim, distance, dtype, device)
        if directory is not None:
            os.makedirs(directory, exist_ok=True)
            col._write_meta()
            open(os.path.join(directory, "wal.jsonl"), "w").close()
        return col

    @staticmethod
    def _snapshot_dir(directory: str):
        """-> (snapshot number, directory holding points.json + vectors.npy) of the current snapshot, or (0, None).
        ``CURRENT`` names the snapshot; a collection written by an older build has the two files next to meta.json."""
        cur = os.path.join(directory, "CURRENT")
        if os.path.exists(cur):
            with open(cur, encoding="utf-8") as f:
                no = int(f.read().strip() or 0)
            d = os.path.join(directory, f"snap-{no}")
            if no > 0 and os.path.isdir(d):
                return no, d
            raise RuntimeError(f"collection at {directory!r}: CURRENT names snapshot {no}, which does not exist")
        if os.path.exists(os.path.join(directory, "points.json")) and os.path.exists(os.path.join(directory, "vectors.npy")):
            return 0, directory
        return 0, None

    @classmethod
    def open(cls, directory: str, device: int):
        with open(cls.meta_path(directory), encoding="utf-8") as f:
            meta = json.load(f)
        col = cls(directory, meta["name"], meta["dim"], meta["distance"], meta.get("dtype", "f32"), device)
        col._snap_no, sdir = cls._snapshot_dir(directory)
        if sdir is not None:
            with open(os.path.join(sdir, "points.json"), encoding="utf-8") as f:
                pts = json.load(f)
            vec = np.load(os.path.join(sdir, "vectors.npy"), mmap_mode="r")   # paged in when the gallery is materialised
            if vec.shape != (len(pts), col.dim):
                raise RuntimeError(f"collection {col.name!r}: snapshot shape {vec.shape} != ({len(pts)}, {col.dim})")
            for pid, payload in pts:
                col._add_point(pid if isinstance(pid, int) else str(pid), payload)
            col.snapshot_vectors = vec
            col.snap_src = np.arange(len(pts), dtype=np.int64)
        col._replay_wal()
        return col

    def _replay_wal(self) -> None:
        """Applies wal.jsonl strictly in log order on the host (no device needed): upserts are staged, deletes take
        effect at once -- a later upsert of the same id is a new point.  A torn tail (interrupted append) is cut off
        the file, so the next append starts on a fresh line and later records are never glued to garbage."""
        wal = os.path.join(self.directory, "wal.jsonl")
        if not os.path.exists(wal):
            return
        good_end = 0
        needs_newline = False
        with open(wal, "rb") as f:
            data = f.read()
        pos = 0
        while pos < len(data):
            nl = data.find(b"\n", pos)
            end = len(data) if nl < 0 else nl + 1
            line = data[pos:end].strip()
            if line:
                try:
                    rec = json.loads(line.decode("utf-8"))
                    if rec.get("op") == "upsert":
                        vec = np.frombuffer(base64.b64decode(rec["vec"]), dtype=np.float32)
                        if vec.shape[0] != self.dim:
                            raise ValueError("vector length")
                        self._stage(rec["id"], vec, rec["payload"])
                    elif rec.get("op") == "delete":
                        self._delete_host(rec["id"])
                except (ValueError, KeyError, UnicodeDecodeError):
                    break      # torn or corrupt record: everything from here on is dropped
                needs_newline = nl < 0
            good_end = end
            pos = end
        if good_end < len(data) or needs_newline:
            with open(wal, "r+b") as f:
                f.truncate(good_end)
                if needs_newline:
                    f.seek(good_end)
                    f.write(b"\n")

    def _write_meta(self) -> None:
        meta = {"name": self.name, "dim": self.dim, "distance": self.distance, "dtype": self.dtype,
                "format": FORMAT_VERSION}
        tmp = self.meta_path(self.directory) + ".tmp"
        with open(tmp, "w", encoding="utf-8") as f:
            json.dump(meta, f)
        os.replace(tmp, self.meta_path(self.directory))

    def _wal_append(self, rec: dict) -> None:
        if self.directory is None:
            return
        if self._wal is None:
            self._wal = open(os.path.join(self.directory, "wal.jsonl"), "a", encoding="utf-8")
        self._wal.write(json.dumps(rec, separators=(",", ":")) + "\n")
        self._wal.flush()

    def save(self) -> None:
        """Snapshot stored vectors + points and truncate the WAL (needs the device copy).  The snapshot is one unit:
        both files are written into a fresh ``snap-<N>`` directory, which becomes current by an atomic rename of the
        ``CURRENT`` pointer; a crash at any point leaves either the old snapshot with the whole WAL or the new one
        (whose WAL records, if still there, replay to the same state)."""
        if self.directory is None or not self._dirty:
            return
        if self.gallery is None:
            return  # nothing materialised in this process: the WAL already holds every change
        vec = self.stored_vectors(range(len(self.ids))) if self.ids else np.zeros((0, self.dim), np.float32)
        no = self._snap_no + 1
        sdir = os.path.join(self.directory, f"snap-{no}")
        if os.path.isdir(sdir):
            shutil.rmtree(sdir)           # left behind by a crash before its CURRENT switch
        os.makedirs(sdir)
        with open(os.path.join(sdir, "vectors.npy"), "wb") as f:
            np.save(f, vec)
            f.flush()
            os.fsync(f.fileno())
        with open(os.path.join(sdir, "points.json"), "w", encoding="utf-8") as f:
            json.dump([[pid, pl] for pid, pl in zip(self.ids, self.payloads)], f)
            f.flush()
            os.fsync(f.fileno())
        tmp = os.path.join(self.directory, "CURRENT.tmp")
        with open(tmp, "w", encoding="utf-8") as f:
            f.write(str(no))
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, os.path.join(self.directory, "CURRENT"))
        if self._wal is not None:
            self._wal.close()
            self._wal = None
        open(os.path.join(self.directory, "wal.jsonl"), "w").close()
        old = os.path.join(self.directory, f"snap-{self._snap_no}")
        self._snap_no = no
        if os.path.isdir(old):
            shutil.rmtree(old, ignore_errors=True)
        for legacy in ("vectors.npy", "points.json"):
            try:
                os.unlink(os.path.join(self.directory, legacy))
            except FileNotFoundError:
                pass
        self._dirty = False

    def close(self) -> None:
        try:
            self.save()
        finally:
            if self._wal is not None:
                self._wal.close()
                self._wal = None
            if self.gallery is not None:
                self.gallery.close()
                self.gallery = None

    # ------------------------------------------------------------------ points
    def __len__(self) -> int:
        return len(self.ids)

    def _index_add(self, slot: int, payload: dict) -> None:
        for key, value in payload.items():
            if isinstance(value, (list, tuple)):
                self.list_keys.add(key)
            values = value if isinstance(value, (list, tuple)) else [value]
            for v in values:
                if _indexable(v):
                    self.index.setdefault(key, {}).setdefault(_vkey(v), set()).add(slot)

    def _index_remove(self, slot: int, payload: dict) -> None:
        for key, value in payload.items():
            values = value if isinstance(value, (list, tuple)) else [value]
            for v in values:
                if _indexable(v):
                    s = self.index.get(key, {}).get(_vkey(v))
                    if s is not None:
                        s.discard(slot)

    def _add_point(self, pid, payload: Optional[dict]) -> int:
        payload = copy.deepcopy(payload) if payload else {}
        slot = self.slot_of.get(pid)
        if slot is None:
            slot = len(self.ids)
            self.ids.append(pid)
            self.payloads.append(payload)
            self.slot_of[pid] = slot
            self._order = None
        else:
            self._index_remove(slot, self.payloads[slot])
            self.payloads[slot] = payload
        self._index_add(slot, payload)
        self._columns_n = -1
        return slot

    def _stage(self, pid, vec: np.ndarray, payload: Optional[dict]) -> int:
        slot = self._add_point(pid, payload)
        self.pending[slot] = np.array(vec, dtype=np.float32, copy=True)
        self._dirty = True
        return slot

    def upsert(self, pid, vector, payload: Optional[dict]) -> None:
        pid = canonical_id(pid)
        vec = np.asarray(vector, dtype=np.float32).reshape(-1)
        if vec.shape[0] != self.dim:
            raise ValueError(f"Wrong input: Vector dimension error: expected dim: {self.dim}, got {vec.shape[0]}")
        if payload is not None and not isinstance(payload, dict):
            raise ValueError("payload must be a dict or None")
        self._wal_append({"op": "upsert", "id": pid, "payload": payload or {},
                          "vec": base64.b64encode(vec.tobytes()).decode("ascii")})
        self._stage(pid, vec, payload)
        if len(self.pending) >= _FLUSH_THRESHOLD:
            self.flush()

    def upsert_many(self, pids: Sequence, vectors: np.ndarray, payloads: Optional[Sequence[Optional[dict]]]) -> None:
        for i, pid in enumerate(pids):
            self.upsert(pid, vectors[i], None if payloads is None else payloads[i])

    def upsert_device(self, pids: Sequence, vectors, payloads: Optional[Sequence[Optional[dict]]]) -> None:
        """Bulk upsert of embeddings that already live on the GPU (torch CUDA tensor [n, dim], any float dtype):
        rows go straight into K1 by device pointer.  They are not journalled row by row -- the next ``save()``
        (client.close / interpreter exit) snapshots them."""
        n = len(pids)
        if tuple(vectors.shape) != (n, self.dim):
            raise ValueError(f"Wrong input: Vector dimension error: expected [{n}, {self.dim}], got {tuple(vectors.shape)}")
        self.flush()                       # keep slot order: earlier staged points reach the device first
        canon = [canonical_id(p) for p in pids]
        if len(set(canon)) != n:
            raise ValueError("duplicate point ids in one upsert_device call")
        slots = np.empty(n, dtype=np.int64)
        for i, pid in enumerate(canon):
            slots[i] = self._add_point(pid, None if payloads is None else payloads[i])
        import torch

        self._ensure_gallery().upsert(vectors.detach().to(torch.float32).contiguous(), slots=slots)
        self._dirty = True

    # ------------------------------------------------------------------ device
    def _ensure_gallery(self):
        if self.gallery is None:
            from .gallery import Gallery

            metric = {"Cosine": "cosine", "Dot": "dot", "Euclid": "euclid", "Manhattan": "manhattan"}[self.distance]
            self.gallery = Gallery(self.dim, dtype=self.dtype, metric=metric, capacity=max(len(self.ids), 1024),
                                   device=self.device)
            if self.dtype in ("bf16", "bfloat16") and os.environ.get("RBOD_BF16_SHADOW", "0") == "1":
                self.gallery.set_option("shadow16", 1)    # fp16 search operand: tighter certification, 2x memory
            if self.snapshot_vectors is not None and self.snap_src is not None and len(self.snap_src):
                # the snapshot file is memory-mapped: stream it to the device in 256 MB pieces (stored form, no K1
                # normalisation), so reopening a large collection never holds a second copy in host memory.  Slots
                # whose vector was re-upserted since (snap_src < 0) get a placeholder row here and their staged
                # vector in the flush that follows; deletes replayed from the WAL have already permuted snap_src.
                src = self.snap_src
                identity = len(src) <= len(self.snapshot_vectors) and bool((src == np.arange(len(src))).all())
                step = max(1, (256 << 20) // (4 * self.dim))
                for a in range(0, len(src), step):
                    if identity:
                        rows = self.snapshot_vectors[a:a + step]
                    else:
                        rows = self.snapshot_vectors[np.maximum(src[a:a + step], 0)]
                    self.gallery.upsert(np.ascontiguousarray(rows, dtype=np.float32), raw=True)
            self.snapshot_vectors = None
            self.snap_src = None
        return self.gallery

    def flush(self) -> None:
        """Pushes staged upserts to the GPU in one K1 launch (snapshot rows go first, untouched)."""
        g = self._ensure_gallery()
        if self.pending:
            slots = np.fromiter(sorted(self.pending), dtype=np.int64, count=len(self.pending))
            rows = np.stack([self.pending[int(s)] for s in slots])
            g.upsert(rows, slots=slots)
            self.pending.clear()

    def stored_vectors(self, slots: Iterable[int]) -> np.ndarray:
        """Stored (normalised) float32 vectors of the given slots, from the device."""
        slots = np.fromiter(slots, dtype=np.int64)
        if len(slots) == 0:
            return np.zeros((0, self.dim), dtype=np.float32)
        self.flush()
        return self.gallery.get_rows(slots)

    def _delete_host(self, pid) -> bool:
        """Delete before the gallery exists (WAL replay): the same swap-with-last as ``_delete_now``, applied to the
        host-side vector sources -- staged vectors and the slot -> snapshot-row map -- instead of device rows."""
        assert self.gallery is None
        slot = self.slot_of.get(pid)
        if slot is None:
            return False
        last = len(self.ids) - 1
        n_snap = 0 if self.snap_src is None else len(self.snap_src)
        self._index_remove(slot, self.payloads[slot])
        self.pending.pop(slot, None)
        if slot != last:
            moved = self.ids[last]
            self._index_remove(last, self.payloads[last])
            self.ids[slot], self.payloads[slot] = moved, self.payloads[last]
            self.slot_of[moved] = slot
            self._index_add(slot, self.payloads[slot])
            if last in self.pending:
                self.pending[slot] = self.pending.pop(last)
                if slot < n_snap:
                    self.snap_src[slot] = -1
            elif slot < n_snap and last < n_snap:
                self.snap_src[slot] = self.snap_src[last]
        if last < n_snap:
            self.snap_src = self.snap_src[:last].copy()
        self.ids.pop()
        self.payloads.pop()
        del self.slot_of[pid]
        self._order = None
        self._columns_n = -1
        self._dirty = True
        return True

    def _delete_now(self, pid) -> bool:
        slot = self.slot_of.get(pid)
        if slot is None:
            return False
        last = len(self.ids) - 1
        self._index_remove(slot, self.payloads[slot])
        if slot != last:
            row = self.gallery.get_rows(np.array([last], dtype=np.int64))
            self.gallery.upsert(row, slots=np.array([slot], dtype=np.int64), raw=True)
            moved = self.ids[last]
            self._index_remove(last, self.payloads[last])
            self.ids[slot], self.payloads[slot] = moved, self.payloads[last]
            self.slot_of[moved] = slot
            self._index_add(slot, self.payloads[slot])
        self.ids.pop()
        self.payloads.pop()
        del self.slot_of[pid]
        self.gallery.truncate(last)
        self._order = None
        self._columns_n = -1
        self._dirty = True
        return True

    def delete(self, pids: Iterable) -> int:
        self.flush()
        n = 0
        for pid in pids:
            pid = canonical_id(pid)
            if pid in self.slot_of:
                self._wal_append({"op": "delete", "id": pid})
                n += int(self._delete_now(pid))
        return n

    # ------------------------------------------------------------------ filters / scroll
    def ordered_slots(self) -> List[int]:
        if self._order is None:
            self._order = sorted(range(len(self.ids)), key=lambda s: id_sort_key(self.ids[s]))
        return self._order

    def _match_slots(self, cond) -> Set[int]:
        """Slots satisfying one condition object (duck-typed on the qdrant_client.models classes)."""
        if hasattr(cond, "must") or hasattr(cond, "should") or hasattr(cond, "must_not"):
            res = self.filter_slots(cond)
            return set(range(len(self.ids))) if res is None else res
        if hasattr(cond, "has_id"):
            out = set()
            for pid in cond.has_id:
                s = self.slot_of.get(canonical_id(pid))
                if s is not None:
                    out.add(s)
            return out
        if hasattr(cond, "is_null"):
            key = cond.is_null.key if hasattr(cond.is_null, "key") else cond.is_null
            return {s for s, p in enumerate(self.payloads) if key in p and p[key] is None}
        if hasattr(cond, "is_empty"):
            key = cond.is_empty.key if hasattr(cond.is_empty, "key") else cond.is_empty
            return {s for s, p in enumerate(self.payloads) if p.get(key) in (None, [], ())}
        key = getattr(cond, "key", None)
        if key is None:
            raise ValueError(f"unsupported filter condition {cond!r}")
        match = getattr(cond, "match", None)
        rng = getattr(cond, "range", None)
        if match is not None:
            by_value = self.index.get(key, {})
            if hasattr(match, "value"):
                if match.value is None:
                    return set()
                return set(by_value.get(_vkey(match.value), ()))
            if hasattr(match, "any"):
                out: Set[int] = set()
                for v in match.any:
                    out |= by_value.get(_vkey(v), set())
                return out
            if hasattr(match, "except_"):
                banned: Set[int] = set()
                for v in match.except_:
                    banned |= by_value.get(_vkey(v), set())
                have = set()
                for s in by_value.values():
                    have |= s
                return have - banned
            if hasattr(match, "text"):
                return {s for s, p in enumerate(self.payloads) if isinstance(p.get(key), str) and match.text in p[key]}
            raise ValueError(f"unsupported match {match!r}")
        if rng is not None:
            def ok(v):
                if isinstance(v, bool) or not isinstance(v, (int, float)):
                    return False
                for name, op in (("gt", lambda a, b: a > b), ("gte", lambda a, b: a >= b),
                                 ("lt", lambda a, b: a < b), ("lte", lambda a, b: a <= b)):
                    bound = getattr(rng, name, None)
                    if bound is not None and not op(v, bound):
                        return False
                return True
            return {s for s, p in enumerate(self.payloads) if ok(p.get(key))}
        raise ValueError(f"filter condition on {key!r} has neither match nor range")

    def filter_slots(self, flt) -> Optional[Set[int]]:
        """Set of slots passing ``flt`` (None = no filter = every slot)."""
        if flt is None:
            return None
        result: Optional[Set[int]] = None
        must = getattr(flt, "must", None) or []
        should = getattr(flt, "should", None) or []
        must_not = getattr(flt, "must_not", None) or []
        for group in (must, should, must_not):
            if not isinstance(group, (list, tuple)):
                raise ValueError("filter clauses must be lists of conditions")
        for cond in must:
            s = self._match_slots(cond)
            result = s if result is None else (result & s)
            if not result:
                return set()
        if should:
            any_of: Set[int] = set()
            for cond in should:
                any_of |= self._match_slots(cond)
            result = any_of if result is None else (result & any_of)
        if must_not:
            if result is None:
                result = set(range(len(self.ids)))
            for cond in must_not:
                result -= self._match_slots(cond)
        return result

    def scroll(self, flt=None, limit: int = 10, offset=None):
        """-> (slots of this page in id order, next_page_offset id or None)."""
        allowed = self.filter_slots(flt)
        order = self.ordered_slots()
        start = 0
        if offset is not None:
            key = id_sort_key(canonical_id(offset))
            lo, hi = 0, len(order)
            while lo < hi:
                mid = (lo + hi) // 2
                if id_sort_key(self.ids[order[mid]]) < key:
                    lo = mid + 1
                else:
                    hi = mid
            start = lo
        page: List[int] = []
        nxt = None
        for s in order[start:]:
            if allowed is not None and s not in allowed:
                continue
            if len(page) == limit:
                nxt = self.ids[s]
                break
            page.append(s)
        return page, nxt

    def row_mask(self, allowed: Optional[Set[int]]) -> Optional[np.ndarray]:
        """uint32 bitmask over row slots for the device search (None = all rows)."""
        if allowed is None:
            return None
        n = len(self.ids)
        bits = np.zeros((n + 31) // 32 * 32, dtype=np.uint8)
        if allowed:
            bits[np.fromiter(allowed, dtype=np.int64)] = 1
        return np.packbits(bits, bitorder="little").view(np.uint32).copy()

    def _column(self, key: str):
        """Dictionary-encoded payload column: int32 code per slot (-1 = missing / None / not a scalar)."""
        if self._columns_n != len(self.ids):
            self._columns = {}
            self._columns_n = len(self.ids)
        col = self._columns.get(key)
        if col is None:
            codes = np.full(len(self.ids), -1, dtype=np.int32)
            table: Dict[Any, int] = {}
            for slot, p in enumerate(self.payloads):
                v = p.get(key)
                if _indexable(v):
                    codes[slot] = table.setdefault(_vkey(v), len(table))
            col = (codes, table)
            self._columns[key] = col
        return col

    def group_rows(self, key: str, flt=None):
        """Rows grouped by the scalar payload value under ``key`` (the per-class loop of 32_…py:119-156 as one CSR):
        -> (group values sorted by (type name, value), row slots [n] grouped in that order and in id order inside a
        group, offsets [G+1]).  Rows whose value is None / missing / not a scalar belong to no group.  Vectorised over
        the dictionary-encoded column, so a million labelled rows group in milliseconds."""
        n = len(self.ids)
        codes, table = self._column(key)
        allowed = np.ones(n, dtype=bool)
        if flt is not None:
            words = self.filter_mask(flt)
            allowed = np.unpackbits(words.view(np.uint8), bitorder="little")[:n].astype(bool)
        order = np.fromiter(self.ordered_slots(), dtype=np.int64, count=n)
        sel = order[(codes[order] >= 0) & allowed[order]]
        present = np.unique(codes[sel])
        by_code = {code: vk for vk, code in table.items()}
        names_vk = sorted((by_code[int(c)] for c in present), key=lambda vk: (vk[0], vk[1]))
        rank = np.full(len(table) + 1, -1, dtype=np.int64)
        for r, vk in enumerate(names_vk):
            rank[table[vk]] = r
        r_sel = rank[codes[sel]]
        o = np.argsort(r_sel, kind="stable")
        offsets = np.zeros(len(names_vk) + 1, dtype=np.int64)
        np.cumsum(np.bincount(r_sel, minlength=len(names_vk)), out=offsets[1:])
        return [vk[1] for vk in names_vk], sel[o], offsets

    def filter_mask(self, flt) -> Optional[np.ndarray]:
        """Filter -> uint32 row bitmask for the device search (SURVEY.md §8 f1).  The filters the reference issues
        (AND of payload equalities, 32:125-129, 33:98-103,117-137) compile to vectorised compares over
        dictionary-encoded columns; anything else goes through the general evaluator."""
        if flt is None:
            return None
        must = getattr(flt, "must", None) or []
        # a key that ever held a list matches per element (as Qdrant's MatchValue does on arrays): the dictionary-encoded
        # column holds one code per row and cannot express that, so such filters take the general evaluator
        simple = (not (getattr(flt, "should", None) or []) and not (getattr(flt, "must_not", None) or []) and
                  all(getattr(c, "key", None) is not None and hasattr(getattr(c, "match", None), "value")
                      and getattr(c, "range", None) is None and c.key not in self.list_keys for c in must))
        if not simple:
            return self.row_mask(self.filter_slots(flt))
        n = len(self.ids)
        allowed = np.ones(n, dtype=bool)
        for cond in must:
            codes, table = self._column(cond.key)
            value = cond.match.value
            code = table.get(_vkey(value)) if _indexable(value) else None
            if code is None:
                allowed[:] = False
                break
            allowed &= codes == code
        bits = np.zeros((n + 31) // 32 * 32, dtype=np.uint8)
        bits[:n] = allowed
        return np.packbits(bits, bitorder="little").view(np.uint32).copy()

    def search(self, queries: np.ndarray, k: int, flt=None, filters=None):
        """-> (scores [Q,k] float32, slots [Q,k] int64) via the device (K3 + exact rescoring).  ``flt`` filters every
        query; ``filters`` is one filter (or None) per query instead, all answered in one device search."""
        self.flush()
        q = np.ascontiguousarray(queries, dtype=np.float32)
        if filters is not None:
            if flt is not None:
                raise ValueError("search: pass one filter for all queries or one per query, not both")
            filters = list(filters)
            if len(filters) != len(q):
                raise ValueError(f"search: {len(filters)} filters for {len(q)} queries")
            masks, ids = self._filter_masks(filters)
            if masks is not None:
                res = self.gallery.search(q, k, row_mask=masks, mask_of_query=ids)
                return res.scores, res.rows
        res = self.gallery.search(q, k, row_mask=self.filter_mask(flt))
        return res.scores, res.rows

    def search_mmr(self, queries: np.ndarray, limit: int, candidates: int, diversity, score_thresholds=None,
                   filters=None):
        """Maximal marginal relevance (``Gallery.search_mmr``, kernel K8) of every query, in one device call: ``limit``
        picks among the exact top-``candidates``, in selection order.  ``diversity`` / ``score_thresholds``: one value
        or one per query (a threshold None = none); ``filters``: None or one filter (or None) per query.
        -> (scores [Q, limit] float32, slots [Q, limit] int64)."""
        self.flush()
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        thr = None
        if score_thresholds is not None:
            thr = np.asarray([np.nan if t is None else float(t)
                              for t in np.broadcast_to(np.asarray(score_thresholds, dtype=object), (len(q),))],
                             dtype=np.float32)
        masks, ids = self._filter_masks(list(filters) if filters is not None else [None] * len(q))
        res = self.gallery.search_mmr(q, int(limit), int(candidates), diversity, score_threshold=thr,
                                      row_mask=masks, mask_of_query=None if masks is None else ids)
        return np.asarray(res.scores), np.asarray(res.rows)

    def _filter_masks(self, filters):
        """One filter (or None) per request -> (row masks [M, words], or None when every filter is None; mask id per
        request, int32, -1 = no filter).  Equal filters compile to one mask; models are not hashable, their repr is
        deterministic."""
        masks, mask_id = [], {}
        ids = np.full(len(filters), -1, dtype=np.int32)
        for i, f in enumerate(filters):
            if f is not None:
                key = repr(f)
                if key not in mask_id:
                    mask_id[key] = len(masks)
                    masks.append(self.filter_mask(f))
                ids[i] = mask_id[key]
        return (np.stack(masks) if masks else None), ids

    def recommend(self, requests, strategy: str):
        """Recommendation: ``requests`` = [(positive, negative, filter, k)], where every example is a point id or a raw
        vector and k = limit + offset.  Examples given by id take their stored vector and never appear in that
        request's answer.  ``strategy``:

        * "average_vector": one search of mean(P), or 2 mean(P) - mean(N) when there are negatives, composed in float64
          and rounded to float32 once; scores are the collection's ordinary search scores.  Needs a positive.
        * "best_score": ``Gallery.recommend`` (exact fp64 sweep, kernel K6); scores are larger-is-better for every
          metric (see include/rbod.h, rbod_recommend).

        Each request fetches k + (its distinct example ids) rows, at most 1024, and has 1 to 32 examples.  Requests
        with the same fetch share one device call.  -> [(scores float32, slots int64)] per request, at most k each,
        example points removed."""
        if strategy not in ("average_vector", "best_score"):
            raise ValueError(f"unknown recommend strategy {strategy!r}")
        self.flush()
        plans = []
        for pos, neg, flt, k in requests:
            items = [(x, 1) for x in (pos or [])] + [(x, -1) for x in (neg or [])]
            if not 1 <= len(items) <= MAX_RECOMMEND_EXAMPLES:
                raise ValueError(f"recommend: a request needs 1 to {MAX_RECOMMEND_EXAMPLES} examples, got {len(items)}")
            if strategy == "average_vector" and not pos:
                raise ValueError("recommend: the average_vector strategy needs at least one positive example")
            vecs, ex_slots = self._resolve_examples([x for x, _ in items], "recommend")
            signs = [sign for _, sign in items]
            fetch = int(k) + len(ex_slots)
            if fetch > MAX_RECOMMEND_FETCH:
                raise ValueError(f"recommend: limit + offset + example ids = {fetch} exceeds {MAX_RECOMMEND_FETCH}")
            plans.append((vecs, signs, ex_slots, flt, int(k), fetch))
        stored = self._stored_examples([p[0] for p in plans])
        out = [(np.zeros(0, np.float32), np.zeros(0, np.int64))] * len(plans)
        by_fetch = {}
        for i, p in enumerate(plans):
            if p[4] >= 1:
                by_fetch.setdefault(p[5], []).append(i)
        for fetch, members in by_fetch.items():
            flts = [plans[i][3] for i in members]
            ex = [np.stack([stored[v] if isinstance(v, int) else v for v in plans[i][0]]) for i in members]
            if strategy == "average_vector":
                q = []
                for i, e in zip(members, ex):
                    sg = np.asarray(plans[i][1])
                    e64 = e.astype(np.float64)
                    mp = e64[sg > 0].mean(axis=0)
                    q.append(2.0 * mp - e64[sg < 0].mean(axis=0) if (sg < 0).any() else mp)
                scores, rows = self.search(np.stack(q).astype(np.float32), fetch, filters=flts)
            else:
                masks, ids = self._filter_masks(flts)
                offsets = np.zeros(len(members) + 1, dtype=np.int64)
                np.cumsum([len(e) for e in ex], out=offsets[1:])
                signs = np.concatenate([np.asarray(plans[i][1], dtype=np.int8) for i in members])
                res = self.gallery.recommend(np.concatenate(ex), signs, offsets, fetch,
                                             row_mask=masks, mask_of_request=None if masks is None else ids)
                scores, rows = res.scores, res.rows
            scores, rows = np.asarray(scores), np.asarray(rows)
            for j, i in enumerate(members):
                keep = ~np.isin(rows[j], list(plans[i][2]))
                out[i] = (scores[j][keep][:plans[i][4]], rows[j][keep][:plans[i][4]])
        return out


    def _resolve_examples(self, examples, who: str):
        """Examples of a recommendation or discovery request, each a point id or a raw vector -> (one entry per
        example: the point's slot (int) or the vector as float32 [dim]; the set of slots given by id).  An unknown id
        is a ValueError that names it."""
        vecs, ex_slots = [], set()
        for x in examples:
            if isinstance(x, (str, uuid.UUID)) or (isinstance(x, (int, np.integer)) and not isinstance(x, bool)):
                pid = canonical_id(x)
                slot = self.slot_of.get(pid)
                if slot is None:
                    raise ValueError(f"{who}: point {pid!r} not found in collection {self.name!r}")
                ex_slots.add(slot)
                vecs.append(slot)
            else:
                v = np.asarray(x, dtype=np.float32).reshape(-1)
                if v.shape[0] != self.dim:
                    raise ValueError(f"Wrong input: Vector dimension error: expected dim: {self.dim}, got {v.shape[0]}")
                vecs.append(v)
        return vecs, ex_slots

    def _stored_examples(self, vec_lists):
        """{slot: stored vector} of every slot in the ``_resolve_examples`` lists ``vec_lists``, read in one call."""
        id_slots = sorted({v for vecs in vec_lists for v in vecs if isinstance(v, int)})
        return dict(zip(id_slots, self.stored_vectors(id_slots)))

    def discover(self, requests):
        """Discovery and context search: ``requests`` = [(target, pairs, filter, k)], where ``target`` is None or an
        example, ``pairs`` a list of (positive, negative) examples, every example a point id or a raw vector, and k =
        limit + offset.  ``Gallery.discover`` (exact fp64 sweep, kernel K7) answers them; scores are larger-is-better
        for every metric (see include/rbod.h, rbod_discover).  Examples given by id take their stored vector and never
        appear in that request's answer.

        Each request has a target or at least one pair, 1 to 32 examples, and fetches k + (its distinct example ids)
        rows, at most 1024.  Requests with the same fetch share one device call.  -> [(scores float32, slots int64)]
        per request, at most k each, example points removed."""
        self.flush()
        plans = []
        for target, pairs, flt, k in requests:
            pairs = list(pairs or [])
            items = ([] if target is None else [(target, 0)]) + [(x, r) for p, n in pairs for x, r in ((p, 1), (n, -1))]
            if not items:
                raise ValueError("discover: a request needs a target or at least one context pair")
            if len(items) > MAX_RECOMMEND_EXAMPLES:
                raise ValueError(f"discover: a request has at most {MAX_RECOMMEND_EXAMPLES} examples (a target and "
                                 f"two per pair), got {len(items)}")
            vecs, ex_slots = self._resolve_examples([x for x, _ in items], "discover")
            fetch = int(k) + len(ex_slots)
            if fetch > MAX_RECOMMEND_FETCH:
                raise ValueError(f"discover: limit + offset + example ids = {fetch} exceeds {MAX_RECOMMEND_FETCH}")
            plans.append((vecs, [r for _, r in items], ex_slots, flt, int(k), fetch))
        stored = self._stored_examples([p[0] for p in plans])
        out = [(np.zeros(0, np.float32), np.zeros(0, np.int64))] * len(plans)
        by_fetch = {}
        for i, p in enumerate(plans):
            if p[4] >= 1:
                by_fetch.setdefault(p[5], []).append(i)
        for fetch, members in by_fetch.items():
            ex = [np.stack([stored[v] if isinstance(v, int) else v for v in plans[i][0]]) for i in members]
            masks, ids = self._filter_masks([plans[i][3] for i in members])
            offsets = np.zeros(len(members) + 1, dtype=np.int64)
            np.cumsum([len(e) for e in ex], out=offsets[1:])
            roles = np.concatenate([np.asarray(plans[i][1], dtype=np.int8) for i in members])
            res = self.gallery.discover(np.concatenate(ex), roles, offsets, fetch,
                                        row_mask=masks, mask_of_request=None if masks is None else ids)
            scores, rows = np.asarray(res.scores), np.asarray(res.rows)
            for j, i in enumerate(members):
                keep = ~np.isin(rows[j], list(plans[i][2]))
                out[i] = (scores[j][keep][:plans[i][4]], rows[j][keep][:plans[i][4]])
        return out


class StoreRoot:
    """All collections under one directory (one emulated "server"); ``None`` = in-memory."""

    def __init__(self, directory: Optional[str], dtype: str = "f32", device: int = 0):
        self.directory = directory
        self.dtype = dtype
        self.device = device
        self.open_collections: Dict[str, Collection] = {}
        if directory is not None:
            os.makedirs(directory, exist_ok=True)

    def _dir(self, name: str) -> str:
        if not name or "/" in name or "\\" in name or name in (".", ".."):
            raise ValueError(f"invalid collection name {name!r}")
        return os.path.join(self.directory, name)

    def names(self) -> List[str]:
        if self.directory is None:
            return sorted(self.open_collections)
        out = []
        for entry in sorted(os.listdir(self.directory)):
            if os.path.isfile(Collection.meta_path(os.path.join(self.directory, entry))):
                out.append(entry)
        return out

    def exists(self, name: str) -> bool:
        return name in self.names()

    def get(self, name: str) -> Collection:
        col = self.open_collections.get(name)
        if col is not None:
            return col
        if self.directory is None or not os.path.isfile(Collection.meta_path(self._dir(name))):
            raise CollectionNotFound(name)
        col = Collection.open(self._dir(name), self.device)
        self.open_collections[name] = col
        return col

    def create(self, name: str, dim: int, distance: str, dtype: Optional[str] = None) -> Collection:
        if self.exists(name):
            raise ValueError(f"Wrong input: Collection `{name}` already exists!")
        directory = None if self.directory is None else self._dir(name)
        col = Collection.create(directory, name, dim, distance, dtype or self.dtype, self.device)
        self.open_collections[name] = col
        return col

    def delete(self, name: str) -> bool:
        col = self.open_collections.pop(name, None)
        existed = col is not None
        if col is not None:
            col._dirty = False
            col.close()
        if self.directory is not None and os.path.isdir(self._dir(name)):
            shutil.rmtree(self._dir(name))
            existed = True
        return existed

    def rename(self, old: str, new: str) -> None:
        if not self.exists(old):
            raise CollectionNotFound(old)
        if self.exists(new):
            raise ValueError(f"Wrong input: Collection `{new}` already exists!")
        col = self.open_collections.pop(old, None)
        if self.directory is None:
            col.name = new
            self.open_collections[new] = col
            return
        if col is not None:
            col.save()
            col.close()
        os.rename(self._dir(old), self._dir(new))
        with open(Collection.meta_path(self._dir(new)), encoding="utf-8") as f:
            meta = json.load(f)
        meta["name"] = new
        with open(Collection.meta_path(self._dir(new)), "w", encoding="utf-8") as f:
            json.dump(meta, f)

    def close(self) -> None:
        for col in list(self.open_collections.values()):
            col.close()
        self.open_collections.clear()
