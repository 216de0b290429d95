"""The matching service: query embeddings in; identity ids, scores and accept/reject out.

Replaces the inline per-face loop of the reference -
``FaceRecognitionProcessor.recognize_faces`` (infrenceServer.py:530-552) and
``CameraProcessor.process_frame`` (peopleCount.py:860-887) - with one batched call into
libfrg.so.  The two thin classes at the bottom keep the reference's own names, thresholds and
result shapes so a call site can be switched over line for line (INTEGRATION.md).
"""
from __future__ import annotations

import contextlib
import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _native as N
from .gallery import GalleryStore

LIVE_THRESHOLD = 0.4         # infrenceServer.py:407
CAMPUS_THRESHOLD = 0.45      # peopleCount.py:829
CAMPUS_UNKNOWN = 0.35        # peopleCount.py:830


@dataclass
class MatchResult:
    rows: np.ndarray      # int64 [F, k]   gallery rows, -1 = none
    scores: np.ndarray    # fp32  [F, k]   cosine score (or Euclidean distance), -1.0 / +inf = none
    accept: np.ndarray    # bool  [F]      decision on slot 0 at the call's threshold
    ids: Optional[List[List[Optional[str]]]] = None
    variant: str = ""
    launches: int = 0
    layout_version: int = 0      # GalleryStore.layout_version the rows belong to (compact() renumbers rows)


@dataclass
class RangeResult:
    counts: np.ndarray            # int64 [F]   rows at or above the threshold (Euclidean: at or below)
    rows: List[np.ndarray]        # per query: int64, COMPLETE, best first (score desc / distance asc, then row asc)
    scores: List[np.ndarray]      # per query: fp32, exact, in the same order
    ids: Optional[List[List[Optional[str]]]] = None
    variant: str = ""
    layout_version: int = 0


def best_first(rows: np.ndarray, scores: np.ndarray, metric: str = "cosine"):
    """The project's result order over a complete hit list: score desc (distance asc), then row asc."""
    order = np.lexsort((rows, scores if metric == "euclidean" else -scores))
    return rows[order], scores[order]


def range_lists(counts: np.ndarray, rows: np.ndarray, scores: np.ndarray, metric: str = "cosine"):
    """[F, max_hits] gallery-order blocks whose counts all fit -> per-query best-first arrays."""
    out_r, out_s = [], []
    for f, c in enumerate(counts.tolist()):
        r, sc = best_first(rows[f, :c], scores[f, :c], metric)
        out_r.append(r)
        out_s.append(sc)
    return out_r, out_s


def _params(metric: str, variant: str, threshold: float, tenant: int, row_offset: int) -> N.MatchParams:
    return N.MatchParams(N.METRICS[metric], N.VARIANTS[variant], float(np.float32(threshold)),
                         int(tenant), int(row_offset), 0, 0)


def _reading(store):
    """The store's read section (GalleryStore.reading): match + row -> id translation are atomic with respect to
    compact().  Stores without one (sharded galleries never renumber rows; test doubles) need none."""
    fn = getattr(store, "reading", None)
    return fn() if fn is not None else contextlib.nullcontext()


class Matcher:
    """``match(Q)`` for host (numpy) batches, ``match_device(Q)`` for batches already on the GPU."""

    def __init__(self, store: GalleryStore, metric: str = "cosine"):
        self.store = store
        self.metric = metric

    # ---- host buffers in, host buffers out: H2D + kernels + D2H inside one C call
    def match(self, Q: np.ndarray, k: int = 1, threshold: float = LIVE_THRESHOLD,
              company_id: Optional[str] = None, variant: str = "auto", row_offset: int = 0,
              with_ids: bool = True, out: Optional[MatchResult] = None) -> MatchResult:
        Q = np.ascontiguousarray(Q, dtype=np.float32).reshape(-1, self.store.dim)
        F = len(Q)
        if out is None:
            out = MatchResult(np.empty((F, k), np.int64), np.empty((F, k), np.float32), np.zeros(F, np.uint8))
        tenant = -1 if company_id is None else self.store.tenant_code(company_id, create=False)
        p = _params(self.metric, variant, threshold, tenant, row_offset)
        # one read section: a compaction cannot renumber the rows between the match and their translation.
        # With with_ids=False the caller translates later - inside its own `with store.reading():` around this
        # call (the processors below), or checked through `ids_of(rows, layout_version=out.layout_version)`.
        with _reading(self.store):
            out.layout_version = getattr(self.store, "layout_version", 0)
            N.check(N.lib.frg_match_host(self.store.handle, Q.ctypes.data, F, int(k), C.byref(p),
                                         out.rows.ctypes.data, out.scores.ctypes.data,
                                         out.accept.ctypes.data))
            out.variant, out.launches = N.last_variant(), N.last_launch_count()
            if out.accept.dtype != np.bool_:
                out.accept = out.accept.view(np.bool_)
            if with_ids:
                out.ids = self.store.ids_of(out.rows)
        return out

    # ---- device tensors in/out, enqueued on the caller's stream (torch is only the allocator here)
    def match_device(self, Q, k: int = 1, threshold: float = LIVE_THRESHOLD, company_id: Optional[str] = None,
                     variant: str = "auto", row_offset: int = 0, out=None, stream: Optional[int] = None,
                     tenant: Optional[int] = None):
        """tenant: a tag code given directly (sharded galleries keep their own id / tenant tables)."""
        import torch
        assert Q.is_cuda and Q.dtype == torch.float32 and Q.is_contiguous()
        F = Q.shape[0]
        if out is None:
            out = (torch.empty((F, k), dtype=torch.int64, device=Q.device),
                   torch.empty((F, k), dtype=torch.float32, device=Q.device),
                   torch.empty((F,), dtype=torch.uint8, device=Q.device))
        rows, scores, accept = out
        if stream is None:
            stream = torch.cuda.current_stream(Q.device).cuda_stream
        if tenant is None:
            tenant = -1 if company_id is None else self.store.tenant_code(company_id, create=False)
        p = _params(self.metric, variant, threshold, tenant, row_offset)
        N.check(N.lib.frg_match(self.store.handle, C.c_void_p(Q.data_ptr()), F, int(k), C.byref(p),
                                C.c_void_p(rows.data_ptr()), C.c_void_p(scores.data_ptr()),
                                C.c_void_p(accept.data_ptr()), C.c_void_p(stream)))
        return rows, scores, accept

    # ---- one call for a batch whose queries belong to different companies
    def _tenant_codes(self, company_ids, F: int) -> np.ndarray:
        company_ids = list(company_ids)
        if len(company_ids) != F:
            raise ValueError("%d company ids for %d queries" % (len(company_ids), F))
        return np.array([-1 if c is None else self.store.tenant_code(c, create=False) for c in company_ids], np.int32)

    def match_tenants(self, Q: np.ndarray, company_ids: Sequence[Optional[str]], k: int = 1,
                      threshold: float = LIVE_THRESHOLD, variant: str = "auto", with_ids: bool = True) -> MatchResult:
        """``match`` with a company filter PER QUERY: row f of the result equals ``match(Q[f:f+1], k, threshold,
        company_ids[f])`` bit for bit, in the caller's order (None = all companies; an unknown company matches
        nothing).  One frg_match_tenants_host call, one read section for the match and the id lookup."""
        Q = np.asarray(Q)
        if Q.ndim != 2 or Q.shape[1] != self.store.dim:
            raise ValueError("Q must be [queries, %d], got shape %s" % (self.store.dim, Q.shape))
        Q = np.ascontiguousarray(Q, dtype=np.float32)
        F = len(Q)
        tenants = self._tenant_codes(company_ids, F)
        out = MatchResult(np.empty((F, k), np.int64), np.empty((F, k), np.float32), np.zeros(F, np.uint8))
        p = _params(self.metric, variant, threshold, -1, 0)
        with _reading(self.store):
            out.layout_version = getattr(self.store, "layout_version", 0)
            N.check(N.lib.frg_match_tenants_host(self.store.handle, Q.ctypes.data, F, int(k), C.byref(p),
                                                 tenants.ctypes.data, out.rows.ctypes.data, out.scores.ctypes.data,
                                                 out.accept.ctypes.data))
            out.variant, out.launches = N.last_variant(), N.last_launch_count()
            out.accept = out.accept.view(np.bool_)
            if with_ids:
                out.ids = self.store.ids_of(out.rows)
        return out

    def match_tenants_device(self, Q, tenants: Sequence[int], k: int = 1, threshold: float = LIVE_THRESHOLD,
                             variant: str = "auto", out=None, stream: Optional[int] = None):
        """Device tensors in / out on the caller's stream, like ``match_device``; tenants: one tag code per query as
        host ints (-1 = all tenants)."""
        import torch
        assert Q.is_cuda and Q.dtype == torch.float32 and Q.is_contiguous() and Q.dim() == 2
        F = Q.shape[0]
        t = np.ascontiguousarray([int(x) for x in tenants], dtype=np.int32)
        if len(t) != F:
            raise ValueError("%d tenants for %d queries" % (len(t), F))
        if out is None:
            out = (torch.empty((F, k), dtype=torch.int64, device=Q.device),
                   torch.empty((F, k), dtype=torch.float32, device=Q.device),
                   torch.empty((F,), dtype=torch.uint8, device=Q.device))
        rows, scores, accept = out
        if stream is None:
            stream = torch.cuda.current_stream(Q.device).cuda_stream
        p = _params(self.metric, variant, threshold, -1, 0)
        N.check(N.lib.frg_match_tenants(self.store.handle, C.c_void_p(Q.data_ptr()), F, int(k), C.byref(p),
                                        t.ctypes.data, C.c_void_p(rows.data_ptr()), C.c_void_p(scores.data_ptr()),
                                        C.c_void_p(accept.data_ptr()), C.c_void_p(stream)))
        return rows, scores, accept

    # ---- every row whose score reaches the threshold (exact fp32)
    def range_host(self, Q: np.ndarray, threshold: float, tenant: int = -1, max_hits: int = 64, strict: bool = False,
                   variant: str = "auto", row_offset: int = 0):
        """One frg_match_range_host call: (counts int64 [F], rows int64 [F, max_hits], scores fp32 [F, max_hits]),
        the FIRST max_hits hits of every query in gallery order (+ row_offset); counts[f] > max_hits = truncated."""
        Q = np.ascontiguousarray(Q, dtype=np.float32).reshape(-1, self.store.dim)
        F = len(Q)
        counts = np.zeros(F, np.int64)
        rows, scores = np.empty((F, max_hits), np.int64), np.empty((F, max_hits), np.float32)
        p = _params(self.metric, variant, threshold, tenant, row_offset)
        p.flags = N.FIRST_STRICT if strict else 0
        N.check(N.lib.frg_match_range_host(self.store.handle, Q.ctypes.data, F, int(max_hits), C.byref(p),
                                           counts.ctypes.data, rows.ctypes.data, scores.ctypes.data))
        return counts, rows, scores

    def match_range(self, Q: np.ndarray, threshold: float, company_id: Optional[str] = None, max_hits: int = 64,
                    strict: bool = False, variant: str = "auto", with_ids: bool = True) -> RangeResult:
        """Every live row with score >= threshold ('>' when strict; Euclidean: distance <= threshold), as COMPLETE
        best-first lists.  max_hits only sizes the first call: the queries whose count exceeded it are re-run once,
        those queries only, with room for their largest count."""
        Q = np.ascontiguousarray(Q, dtype=np.float32).reshape(-1, self.store.dim)
        tenant = -1 if company_id is None else self.store.tenant_code(company_id, create=False)
        with _reading(self.store):
            layout = getattr(self.store, "layout_version", 0)
            counts, rows, scores = self.range_host(Q, threshold, tenant, max_hits, strict, variant)
            variant_ran = N.last_variant()
            over = np.nonzero(counts > max_hits)[0]
            if len(over):
                c2, r2, s2 = self.range_host(Q[over], threshold, tenant, int(counts[over].max()), strict, variant)
                counts[over] = c2
            lists_r, lists_s = range_lists(np.minimum(counts, max_hits), rows, scores, self.metric)
            for j, f in enumerate(over.tolist()):
                lists_r[f], lists_s[f] = best_first(r2[j, :c2[j]], s2[j, :c2[j]], self.metric)
            out = RangeResult(counts, lists_r, lists_s, variant=variant_ran, layout_version=layout)
            if with_ids:
                out.ids = [self.store.ids_of(r[None, :])[0] if len(r) else [] for r in lists_r]
        return out

    # ---- the gallery against itself: every pair of stored rows a < b at or above the threshold
    def self_join(self, threshold: float, company_id: Optional[str] = None, same_company: bool = False,
                  strict: bool = False, max_hits: int = 16, variant: str = "auto"):
        """Every pair of stored rows a < b with score(a, b) >= threshold ('>' when strict), where score(a, b) is what
        ``match_range`` returns for row b when row a's stored vector is the query.  company_id: only that company's
        rows; same_company: only pairs whose two rows carry the same company tag (every company at once, each within
        itself).  Returns (a int64, b int64, score fp32) arrays ordered by a, then score desc, then b.
        One frg_self_join over the whole store on the device; only the rows that have pairs are copied back, and a row
        with more than max_hits pairs is redone once on its own, with room for its count."""
        import torch
        tenant = -1 if company_id is None else self.store.tenant_code(company_id, create=False)
        p = _params(self.metric, variant, threshold, tenant, 0)
        p.flags = (N.FIRST_STRICT if strict else 0) | (N.JOIN_SAME_TAG if same_company else 0)
        dev = torch.device("cuda", self.store.device)
        none = (np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.float32))

        def run(row0, n, hits):
            counts = torch.empty(n, dtype=torch.int64, device=dev)
            rows = torch.empty((n, hits), dtype=torch.int64, device=dev)
            scores = torch.empty((n, hits), dtype=torch.float32, device=dev)
            N.check(N.lib.frg_self_join(self.store.handle, int(row0), int(n), int(hits), C.byref(p),
                                        C.c_void_p(counts.data_ptr()), C.c_void_p(rows.data_ptr()),
                                        C.c_void_p(scores.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            return counts, rows, scores

        with _reading(self.store), torch.cuda.device(dev):
            n = self.store.rows
            if n == 0:
                return none
            counts, rows, scores = run(0, n, max_hits)
            hit = torch.nonzero(counts).squeeze(1)          # compacted on the device: only these rows come back
            a = hit.cpu().numpy()
            c = counts[hit].cpu().numpy()
            r = rows[hit].cpu().numpy()
            s = scores[hit].cpu().numpy()
            if not len(a):
                return none
            over = c > max_hits
            fit = np.where(over, 0, c)
            keep = np.arange(max_hits)[None, :] < fit[:, None]
            A, B, S = [np.repeat(a, fit)], [r[keep]], [s[keep]]
            for i in np.nonzero(over)[0].tolist():
                c2, r2, s2 = run(int(a[i]), 1, int(c[i]))
                m = min(int(c2.cpu()[0]), int(c[i]))
                A.append(np.full(m, a[i], np.int64))
                B.append(r2[0, :m].cpu().numpy())
                S.append(s2[0, :m].cpu().numpy())
        A, B, S = np.concatenate(A), np.concatenate(B), np.concatenate(S)
        order = np.lexsort((B, -S, A))
        return A[order], B[order], S[order]

    # ---- first row, in gallery order, whose score reaches the threshold (exact fp32)
    def first_above(self, Q: np.ndarray, threshold: float, strict: bool = False, company_id: Optional[str] = None,
                    query_prenormalised: bool = False):
        """(rows int64 [F], scores fp32 [F]); row -1 / score -1.0 when no row qualifies.  The scan rule of
        the enrol-time duplicate check (trainingServer.py:170-200, strict) and of unknown-person
        clustering (peopleCount.py:446-452)."""
        Q = np.ascontiguousarray(Q, dtype=np.float32).reshape(-1, self.store.dim)
        F = len(Q)
        rows, scores = np.empty(F, np.int64), np.empty(F, np.float32)
        tenant = -1 if company_id is None else self.store.tenant_code(company_id, create=False)
        p = _params(self.metric, "scan_f32", threshold, tenant, 0)
        p.flags = (N.FIRST_STRICT if strict else 0) | (N.QUERY_PRENORMALISED if query_prenormalised else 0)
        N.check(N.lib.frg_first_match_host(self.store.handle, Q.ctypes.data, F, C.byref(p),
                                           rows.ctypes.data, scores.ctypes.data))
        return rows, scores


class FaceRecognitionProcessor:
    """Drop-in for the matching half of infrenceServer.FaceRecognitionProcessor (:400-563).

    ``recognize(embeddings, company_id)`` takes the ``face.normed_embedding`` of every detected
    face and returns, per face, what the reference passes to its draw call (:545-558):
    ``person_info`` (metadata, or ``{'name': 'Unknown', 'type': 'unknown'}``), the reported score
    (0 when rejected) and the matched id (None when rejected)."""

    def __init__(self, store, recognition_threshold: float = LIVE_THRESHOLD, matcher=None):
        """store: a ``GalleryStore`` - or a ``ShardedGallery`` together with ``matcher=ShardedMatcher(store)``
        (one process per GPU; every rank makes the same calls)."""
        self.store = store
        self.matcher = matcher if matcher is not None else Matcher(store)
        self._match = getattr(self.matcher, "match_host", None) or self.matcher.match
        self.recognition_threshold = recognition_threshold

    def recognize(self, embeddings: np.ndarray, company_id: Optional[str] = None) -> List[Dict]:
        store = self.store
        if len(embeddings) == 0 or len(store) == 0:      # `if not embeddings: return frame` (:523-525)
            return []
        out = []
        with _reading(store):        # match + id lookup are one read section (compact() renumbers rows)
            r = self._match(embeddings, 1, self.recognition_threshold, company_id, with_ids=False)
            for f in range(len(embeddings)):
                if r.accept[f]:
                    pid = store.id_of(r.rows[f, 0])            # ids only for the faces that matched
                    info = store.metadata(pid) or {"name": pid, "type": "employee"}
                    out.append({"person_id": pid, "person_info": info, "recognition_score": r.scores[f, 0]})
                else:
                    out.append({"person_id": None, "person_info": {"name": "Unknown", "type": "unknown"},
                                "recognition_score": 0})
        return out

    def recognize_frames(self, frames: Sequence) -> List[List[Dict]]:
        """frames: (embeddings, company_id) per frame, each frame of its own company -> one list per frame, equal to
        ``recognize(embeddings, company_id)`` frame by frame, from ONE match_tenants call."""
        frames = list(frames)
        match_tenants = getattr(self.matcher, "match_tenants", None)
        if match_tenants is None:
            raise NotImplementedError("%s has no match_tenants: per-query company filters need a single-GPU Matcher"
                                      % type(self.matcher).__name__)
        embs = []
        for e, _ in frames:
            e = np.asarray(e, dtype=np.float32)
            if e.ndim != 2:
                raise ValueError("embeddings of a frame must be [faces, dim]")
            embs.append(e)
        store = self.store
        if sum(len(e) for e in embs) == 0 or len(store) == 0:
            return [[] for _ in frames]
        Q = np.concatenate([e for e in embs if len(e)], axis=0)
        ids = [c for e, (_, c) in zip(embs, frames) for _ in range(len(e))]
        out, o = [], 0
        with _reading(store):
            r = match_tenants(Q, ids, 1, self.recognition_threshold, with_ids=False)
            for e in embs:
                faces = []
                for f in range(o, o + len(e)):
                    if r.accept[f]:
                        pid = store.id_of(r.rows[f, 0])
                        info = store.metadata(pid) or {"name": pid, "type": "employee"}
                        faces.append({"person_id": pid, "person_info": info, "recognition_score": r.scores[f, 0]})
                    else:
                        faces.append({"person_id": None, "person_info": {"name": "Unknown", "type": "unknown"},
                                      "recognition_score": 0})
                out.append(faces)
                o += len(e)
        return out


class CameraProcessor:
    """Drop-in for the matching half of peopleCount.CameraProcessor (:822-896): three-way decision
    at 0.45 / 0.35 over ALL tenants, and the same stats dict."""

    def __init__(self, store, recognition_threshold: float = CAMPUS_THRESHOLD,
                 unknown_threshold: float = CAMPUS_UNKNOWN, matcher=None):
        self.store = store
        self.matcher = matcher if matcher is not None else Matcher(store)
        self._match = getattr(self.matcher, "match_host", None) or self.matcher.match
        self.recognition_threshold = recognition_threshold
        self.unknown_threshold = unknown_threshold

    def process(self, embeddings: np.ndarray):
        """Returns (events, stats): events[f] is ('recognized', id, float score) |
        ('unknown', None, None) | ('ignored', None, None)."""
        stats = {"faces": 0, "recognized": 0, "unknown": 0}
        store = self.store
        if len(store) == 0:                               # peopleCount.py:850-851
            return [], stats
        stats["faces"] = len(embeddings)
        if len(embeddings) == 0:
            return [], stats
        events = []
        with _reading(store):        # match + id lookup are one read section (compact() renumbers rows)
            r = self._match(embeddings, 1, self.recognition_threshold, with_ids=False)
            # three-way decision in fp32 (peopleCount.py:876-887); ids are looked up only for recognised faces
            accept = r.accept.tolist()
            below = (r.scores[:, 0] < np.float32(self.unknown_threshold)).tolist()   # best_score stays -1 when nothing matched
            rows, scores = r.rows[:, 0].tolist(), r.scores[:, 0].tolist()
            for f in range(len(accept)):
                if accept[f]:
                    events.append(("recognized", store.id_of(rows[f]), scores[f]))
                elif below[f]:
                    events.append(("unknown", None, None))
                else:
                    events.append(("ignored", None, None))
        stats["recognized"] = sum(accept)
        stats["unknown"] = sum(1 for a, b in zip(accept, below) if b and not a)
        return events, stats
