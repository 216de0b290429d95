"""GPU-resident gallery store: the replacement for ``EmbeddingManager.embeddings`` - the
``Dict[str, np.ndarray]`` both reference servers keep in process memory
(infrenceServer.py:48-51, peopleCount.py:706-708).

The device side (libfrg.so) holds, per row, the unit fp32 vector, its bf16 image and an int32 tag
(tenant code, -1 = removed).  The host side, here, keeps what the dict keys and the metadata dict
carried: ``row <-> id string <-> metadata``.  Row order is dict insertion order, because the
reference's strict ``>`` scan resolves exact ties by that order (infrenceServer.py:538-542):

  * a new id appends a row; an existing id is overwritten in place (dict assignment keeps position);
  * a removed id leaves a tombstone; if it is enrolled again later it appends at the END, exactly
    as ``del d[k]; d[k] = v`` does.  ``compact()`` squeezes tombstones out without reordering.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import json
import struct
import threading
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _native as N


class StaleRows(RuntimeError):
    """Row numbers of a match were looked up after ``compact()`` renumbered the gallery."""


class _LayoutLock:
    """Readers-writer lock between matches and ``compact()``.  A match and the row -> id translation of its
    result form ONE read section (many may run at once - the native call releases the GIL); ``compact()``, which
    renumbers rows, is the only writer: it waits for the read sections in flight and holds new ones off while it
    runs.  Without it a match that straddles a compaction has its rows translated through the wrong table and a
    whole batch of accepted faces is attributed to the wrong people.  Read sections nest per thread."""

    def __init__(self):
        self._c = threading.Condition()
        self._readers = 0
        self._writer = False
        self._writers_waiting = 0
        self._depth = threading.local()

    @contextlib.contextmanager
    def read(self):
        d = getattr(self._depth, "n", 0)
        if d == 0:
            with self._c:
                while self._writer or self._writers_waiting:
                    self._c.wait()
                self._readers += 1
        self._depth.n = d + 1
        try:
            yield
        finally:
            self._depth.n = d
            if d == 0:
                with self._c:
                    self._readers -= 1
                    if not self._readers:
                        self._c.notify_all()

    @contextlib.contextmanager
    def write(self):
        if getattr(self._depth, "n", 0):
            raise RuntimeError("compact() inside a read section of the same thread would wait for itself")
        with self._c:
            self._writers_waiting += 1
            while self._writer or self._readers:
                self._c.wait()
            self._writers_waiting -= 1
            self._writer = True
        try:
            yield
        finally:
            with self._c:
                self._writer = False
                self._c.notify_all()


def _ptr(a: Optional[np.ndarray]):
    # the plain address: ndarray.ctypes.data_as() costs ~7 us per call, four of them were a third of a
    # small frame's end-to-end time
    return None if a is None else a.ctypes.data


class GalleryStore:
    def __init__(self, dim: int = 512, capacity: int = 1024, device: int = 0, bf16_plane: bool = True,
                 raw: bool = False, bf16_only: bool = False):
        """bf16_only: keep only the bf16 scan plane (1 KB per 512-d row instead of 3 KB) - the "bf16
        gallery mode": matches return the bf16 filter scores (within the measured bound eps[q] of fp32: ~3.6e-3 for ordinary data, at most 7.9e-3), 100 M rows fit one B200."""
        self.dim = int(dim)
        self.device = int(device)
        self.bf16_only = bool(bf16_only)
        flags = ((N.STORE_BF16_PLANE if bf16_plane else 0) | (N.STORE_RAW if raw else 0) |
                 (N.STORE_BF16_ONLY if bf16_only else 0))
        h = C.c_void_p()
        N.check(N.lib.frg_store_create(self.device, self.dim, int(capacity), flags, C.byref(h)))
        self._h = h
        self._lock = threading.RLock()               # the reference's embeddings_lock
        self._row_of: Dict[str, int] = {}
        self._id_of: Dict[int, str] = {}
        self._meta: Dict[str, Dict] = {}
        self._tenants: Dict[str, int] = {}
        self._tenant_of: Dict[str, int] = {}         # id -> tenant code (company subset sizes without a device read)
        self._anon_tags: Dict[int, int] = {}         # tenant code -> rows filled synthetically with it
        self._anon: List[Tuple[int, int, int]] = []  # (row0, n, global_row0) ranges filled synthetically
        self._rows = 0                               # mirror of stats.rows
        self._layout = _LayoutLock()                 # matches + id lookups (readers) vs compact() (writer)
        self.layout_version = 0                      # bumped by every compact(): row numbers of older results are void

    # ------------------------------------------------------------------ life-cycle
    def close(self):
        if getattr(self, "_h", None):
            N.lib.frg_store_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        if not self._h:
            raise RuntimeError("store is closed")
        return self._h

    # ------------------------------------------------------------------ tenants
    def tenant_code(self, company_id: Optional[str], create: bool = True) -> int:
        """Small int standing for a company id (the tag stored per row).  None -> 0."""
        if company_id is None:
            return 0
        key = str(company_id)
        with self._lock:
            if key not in self._tenants:
                if not create:
                    return 0x7FFFFFFF  # a tag no row carries: matches nothing (negative would mean "all")
                self._tenants[key] = len(self._tenants) + 1
            return self._tenants[key]

    def tenant_keys(self) -> Dict[int, str]:
        """tag code -> company key, for every company this store has given a code."""
        with self._lock:
            return {code: key for key, code in self._tenants.items()}

    # ------------------------------------------------------------------ raw row API
    def stats(self) -> N.StoreStats:
        st = N.StoreStats()
        N.check(N.lib.frg_store_stats(self.handle, C.byref(st)))
        return st

    def reserve(self, capacity: int):
        N.check(N.lib.frg_store_reserve(self.handle, int(capacity)))

    def append_rows(self, vecs: np.ndarray, tags: Optional[np.ndarray] = None, prenormalised: bool = False) -> int:
        vecs = np.ascontiguousarray(vecs, dtype=np.float32).reshape(-1, self.dim)
        t = None if tags is None else np.ascontiguousarray(tags, dtype=np.int32)
        with self._lock:
            first = self._rows
            N.check(N.lib.frg_store_upsert_host(self.handle, None, _ptr(vecs), _ptr(t), len(vecs),
                                                N.ROWS_PRENORMALISED if prenormalised else 0))
            self._rows += len(vecs)
            return first

    def overwrite_rows(self, rows: Sequence[int], vecs: np.ndarray, tags: Optional[np.ndarray] = None,
                       prenormalised: bool = False):
        r = np.ascontiguousarray(rows, dtype=np.int64)
        vecs = np.ascontiguousarray(vecs, dtype=np.float32).reshape(-1, self.dim)
        t = None if tags is None else np.ascontiguousarray(tags, dtype=np.int32)
        with self._lock:
            N.check(N.lib.frg_store_upsert_host(self.handle, _ptr(r), _ptr(vecs), _ptr(t), len(r),
                                                N.ROWS_PRENORMALISED if prenormalised else 0))

    def remove_rows(self, rows: Sequence[int]):
        r = np.ascontiguousarray(rows, dtype=np.int64)
        if len(r):
            with self._lock:
                N.check(N.lib.frg_store_remove_host(self.handle, _ptr(r), len(r)))

    def read_rows(self, row0: int = 0, n: Optional[int] = None):
        with self._lock:
            n = self._rows - row0 if n is None else n
            vecs = np.empty((n, self.dim), np.float32)
            tags = np.empty(n, np.int32)
            N.check(N.lib.frg_store_read_host(self.handle, int(row0), int(n), _ptr(vecs), _ptr(tags)))
            return vecs, tags

    def read_tags(self, row0: int = 0, n: Optional[int] = None) -> np.ndarray:
        """Tags of rows [row0, row0 + n) (company code, -1 = removed), without their vectors."""
        with self._lock:
            n = self._rows - row0 if n is None else n
            tags = np.empty(n, np.int32)
            N.check(N.lib.frg_store_read_host(self.handle, int(row0), int(n), None, _ptr(tags)))
            return tags

    def fill_synthetic(self, n: int, global_row0: int = 0, seed: int = 1234, tag: int = 0, stream=None):
        """Append n rows of the frg-synth-v1 gallery (bench / scale tests; oracle.synth is the CPU twin).
        Their ids are implicit: ``"%024x" % global_row``."""
        with self._lock:
            N.check(N.lib.frg_store_fill_synthetic(self.handle, int(n), int(global_row0), int(seed), int(tag),
                                                   C.c_void_p(stream or 0)))
            self._anon.append((self._rows, int(n), int(global_row0)))
            self._anon_tags[int(tag)] = self._anon_tags.get(int(tag), 0) + int(n)
            self._rows += int(n)

    # ------------------------------------------------------------------ id-level API (the dict)
    def __len__(self):
        with self._lock:
            return len(self._row_of) + sum(n for _, n, _ in self._anon)

    def __contains__(self, pid: str):
        return str(pid) in self._row_of

    @property
    def rows(self) -> int:
        return self._rows

    def ids(self) -> List[str]:
        """Live ids in gallery (= dict) order."""
        with self._lock:
            return [self._id_of[r] for r in sorted(self._id_of)]

    def row_of(self, pid: str) -> int:
        return self._row_of.get(str(pid), -1)

    def id_of(self, row: int) -> Optional[str]:
        row = int(row)
        if row < 0:
            return None
        pid = self._id_of.get(row)
        if pid is not None:
            return pid
        for r0, n, g0 in self._anon:
            if r0 <= row < r0 + n:
                return "%024x" % (g0 + row - r0)
        return None

    def reading(self):
        """Context manager: a match and the translation of its rows (``id_of`` / ``ids_of`` / ``metadata``) belong
        in ONE ``with store.reading():`` block, so that ``compact()`` cannot renumber the rows in between.
        ``Matcher.match(with_ids=True)`` and the two processors do this themselves."""
        return self._layout.read()

    def ids_of(self, rows, layout_version: Optional[int] = None) -> List[List[Optional[str]]]:
        """id_of over a whole [F, k] result (one pass over plain Python ints: ~0.1 us per slot).
        layout_version: the ``MatchResult.layout_version`` the rows belong to - raises :class:`StaleRows` when a
        ``compact()`` has renumbered the gallery since (only possible outside a ``reading()`` block)."""
        if layout_version is not None and layout_version != self.layout_version:
            raise StaleRows("rows of layout %d looked up in layout %d: the gallery was compacted in between"
                            % (layout_version, self.layout_version))
        get, anon = self._id_of.get, self._anon

        def one(r):
            if r < 0:
                return None
            pid = get(r)
            if pid is None:
                for r0, n, g0 in anon:
                    if r0 <= r < r0 + n:
                        return "%024x" % (g0 + r - r0)
            return pid

        rows = np.asarray(rows)
        return [[one(r) for r in rr] for rr in rows.reshape(len(rows), -1).tolist()]

    def metadata(self, pid: str) -> Optional[Dict]:
        return self._meta.get(str(pid))

    def count_tenant(self, company_id: Optional[str]) -> int:
        """Live ids of one company - `len(get_embeddings_for_company(c))` (infrenceServer.py:343-380) - from the
        host-side id table, no device read.  (Synthetic fills count by the tag they were filled with.)"""
        code = self.tenant_code(company_id, create=False)
        with self._lock:
            return sum(1 for c in self._tenant_of.values() if c == code) + self._anon_tags.get(code, 0)

    def upsert(self, ids: Sequence[str], vecs: np.ndarray, company_ids: Optional[Sequence[Optional[str]]] = None,
               meta: Optional[Sequence[Dict]] = None, prenormalised: bool = False):
        """``self.embeddings[id] = v / ||v||`` for a batch, in the given order
        (infrenceServer.py:273,326; peopleCount.py:790,808)."""
        vecs = np.ascontiguousarray(vecs, dtype=np.float32).reshape(-1, self.dim)
        if len(ids) != len(vecs):
            raise ValueError("ids and vecs differ in length")
        with self._lock:
            tags = np.array([self.tenant_code(c) for c in (company_ids or [None] * len(ids))], np.int32)
            # repeated dict assignment: position is fixed by the FIRST occurrence of an id in the
            # batch, content by the LAST
            last = {str(p): i for i, p in enumerate(ids)}
            new_i, old_i = [], []
            for p in dict.fromkeys(str(p) for p in ids):
                (old_i if p in self._row_of else new_i).append(last[p])
            if old_i:
                rows = [self._row_of[str(ids[i])] for i in old_i]
                self.overwrite_rows(rows, vecs[old_i], tags[old_i], prenormalised)
            if new_i:
                first = self.append_rows(vecs[new_i], tags[new_i], prenormalised)
                for j, i in enumerate(new_i):
                    p = str(ids[i])
                    self._row_of[p] = first + j
                    self._id_of[first + j] = p
            for i in old_i + new_i:
                self._tenant_of[str(ids[i])] = int(tags[i])
            if meta is not None:
                for p, m in zip(ids, meta):
                    self._meta[str(p)] = m

    def remove(self, ids: Iterable[str]) -> int:
        """``del self.embeddings[id]`` (infrenceServer.py:248-251).  Unknown ids are ignored."""
        with self._lock:
            rows = []
            for p in ids:
                p = str(p)
                r = self._row_of.pop(p, None)
                if r is not None:
                    rows.append(r)
                    self._id_of.pop(r, None)
                    self._meta.pop(p, None)
                    self._tenant_of.pop(p, None)
            self.remove_rows(rows)
            return len(rows)

    def compact(self):
        """Drop tombstones; order (hence tie behaviour) is unchanged.  Rows are renumbered: waits for every
        match / id lookup in flight (``reading()``), holds new ones off meanwhile, bumps ``layout_version``."""
        with self._layout.write(), self._lock:
            n = self._rows
            mapping = np.empty(n, np.int64)
            N.check(N.lib.frg_store_compact(self.handle, _ptr(mapping)))
            new_row_of, new_id_of = {}, {}
            for p, r in self._row_of.items():
                nr = int(mapping[r])
                new_row_of[p] = nr
                new_id_of[nr] = p
            self._row_of, self._id_of = new_row_of, new_id_of
            self._anon = [(int(mapping[r0]), cnt, g0) for r0, cnt, g0 in self._anon if cnt and mapping[r0] >= 0]
            self._rows = int((mapping >= 0).sum())
            self.layout_version += 1

    def snapshot_arrays(self):
        """(ids, G fp32[n, dim], tags) of the LIVE rows in gallery order - what get_all() returned
        as dict copies (peopleCount.py:816-819).  For tests and export, not for matching."""
        with self._lock:
            vecs, tags = self.read_rows(0, self._rows)
            live = np.nonzero(tags >= 0)[0]
            return [self.id_of(int(r)) for r in live], vecs[live], tags[live]

    # ------------------------------------------------------------------ bulk snapshot (section 8f-3)
    SNAP_MAGIC = b"FRGSNAP1"

    def save(self, path: str, chunk_rows: int = 65536) -> int:
        """Write the LIVE rows, in gallery order, to one file: header, id/tenant/metadata table (JSON),
        int32 tags, raw fp32 unit vectors.  Replaces the reference's one-pickle-blob-per-person in
        GridFS (producer trainingServer.py:383-398; consumers infrenceServer.py:269-271,
        peopleCount.py:786-788): nothing to unpickle, one sequential read, and the vectors reload
        bit for bit (they are stored normalised and re-ingested as such).  Returns the row count."""
        with self._lock:
            n_all = self._rows
            _, tags_all = self.read_rows(0, n_all) if n_all else (None, np.zeros(0, np.int32))
            live = np.nonzero(tags_all >= 0)[0]
            ids = [self.id_of(int(r)) for r in live]
            table = json.dumps({"ids": ids, "tenants": self._tenants,
                                "meta": {i: self._meta[i] for i in ids if i in self._meta}},
                               default=str).encode("utf-8")
            with open(path, "wb") as f:
                f.write(self.SNAP_MAGIC)
                f.write(struct.pack("<IIQQ", self.dim, 0, len(live), len(table)))
                f.write(table)
                f.write(np.ascontiguousarray(tags_all[live], np.int32).tobytes())
                # vectors: contiguous runs of live rows are read back chunk by chunk
                for a in range(0, len(live), chunk_rows):
                    idx = live[a:a + chunk_rows]
                    lo, hi = int(idx[0]), int(idx[-1]) + 1
                    vecs, _ = self.read_rows(lo, hi - lo)
                    f.write(np.ascontiguousarray(vecs[idx - lo], np.float32).tobytes())
            return int(len(live))

    @classmethod
    def load(cls, path: str, device: int = 0, bf16_plane: bool = True, chunk_rows: int = 65536,
             capacity_slack: float = 0.0) -> "GalleryStore":
        """Rebuild a store from :meth:`save` output: rows land in the saved order (so ties resolve as
        before), vectors are ingested as stored (no second normalisation)."""
        with open(path, "rb") as f:
            if f.read(8) != cls.SNAP_MAGIC:
                raise ValueError("%s is not a gallery snapshot" % path)
            dim, _flags, n, tlen = struct.unpack("<IIQQ", f.read(24))
            table = json.loads(f.read(tlen).decode("utf-8"))
            tags = np.frombuffer(f.read(4 * n), dtype=np.int32)
            store = cls(dim=dim, capacity=int(n * (1.0 + capacity_slack)) + 1, device=device, bf16_plane=bf16_plane)
            for a in range(0, n, chunk_rows):
                b = min(n, a + chunk_rows)
                vecs = np.frombuffer(f.read(4 * dim * (b - a)), dtype=np.float32).reshape(b - a, dim)
                store.append_rows(vecs, tags[a:b], prenormalised=True)
        ids = table["ids"]
        store._tenants = {str(k): int(v) for k, v in table["tenants"].items()}
        store._meta = dict(table.get("meta", {}))
        for r, pid in enumerate(ids):
            store._row_of[pid] = r
            store._id_of[r] = pid
            store._tenant_of[pid] = int(tags[r])
        return store
