"""Enrolment-time checks of the reference's embedding worker, on the device gallery
(SURVEY.md section 8f-2; trainingServer.py:170-214).

  * duplicate face:   first stored template of the company, in cursor order, with cos > 0.4
                      (trainingServer.py:170-200) -> one exact scan over the tenant's rows instead of
                      one GridFS fetch + unpickle + np.dot per stored person.
  * same person:      every pair of the <= 3 pose embeddings must have cos >= 0.4
                      (trainingServer.py:202-214).
  * stored template:  plain fp32 mean of the pose embeddings (trainingServer.py:355); the gallery
                      normalises it on ingest.

Which gallery to scan.  The reference's duplicate scan reads the Mongo collection, not the live cache: EVERY
document of the company that has an embeddingId - whatever its status, blacklisted or not - and only the
collection being enrolled into (employees OR visitors, chosen by `id_field`).  The live matching gallery
(`EmbeddingManager.store`) is the wrong thing to scan: it has evicted exactly the inactive / blacklisted people
(infrenceServer.py:234-258) a re-enrolment must still be caught against, and it mixes employees and visitors
under one tenant tag.  Use an :class:`EnrolmentGallery` - every enrolled template, tagged (company, kind),
never evicted - and pass `kind=` to ``check_duplicate_face``.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _native as N
from .gallery import GalleryStore
from .matcher import Matcher, _reading


def enrolment_tenant(company_id: Optional[str], kind: Optional[str]) -> Optional[str]:
    """Tenant key of an enrolment gallery: one tag per (company, collection) - trainingServer.py:174-178 scans
    `collection.find({'companyId': company_id, ...})` of ONE collection."""
    if kind is None:
        return company_id
    return "%s|%s" % ("" if company_id is None else company_id, kind)


class EnrolmentGallery:
    """Every enrolled template of every company, whatever the person's status: what trainingServer.py:170-200
    scans.  A thin id-level wrapper over a ``GalleryStore`` whose tenant tag is (company, kind) and whose
    metadata keeps `doc[id_field]`, the value the reference's check returns (trainingServer.py:191)."""

    def __init__(self, dim: int = 512, capacity: int = 1024, device: int = 0, store: Optional[GalleryStore] = None):
        self.store = store if store is not None else GalleryStore(dim, capacity, device, bf16_plane=False)

    def add(self, doc_ids: Sequence[str], embeddings: np.ndarray, company_ids: Sequence[Optional[str]],
            kinds: Sequence[str], ref_ids: Optional[Sequence] = None):
        """Cursor order = insertion order; an existing document is overwritten in place."""
        meta: List[Dict] = [{"kind": k, "ref_id": (None if ref_ids is None else ref_ids[i])} for i, k in enumerate(kinds)]
        self.store.upsert(list(doc_ids), embeddings, [enrolment_tenant(c, k) for c, k in zip(company_ids, kinds)], meta)

    def remove(self, doc_ids: Sequence[str]) -> int:
        """Only when the DOCUMENT is deleted - never for a status change."""
        return self.store.remove(doc_ids)

    def close(self):
        self.store.close()

SIMILARITY_THRESHOLD = 0.4     # trainingServer.py:70
DUPLICATE_THRESHOLD = 0.4      # trainingServer.py:71


class EnrolmentChecker:
    def __init__(self, store, duplicate_threshold: float = DUPLICATE_THRESHOLD,
                 similarity_threshold: float = SIMILARITY_THRESHOLD, matcher=None):
        """store: a ``GalleryStore``, or a ``ShardedGallery`` with ``matcher=ShardedMatcher(store)`` (the
        duplicate scan then runs on every rank's block and the lowest global row wins; collective)."""
        self.store = store
        self.matcher = matcher if matcher is not None else Matcher(store.store if isinstance(store, EnrolmentGallery) else store)
        self.duplicate_threshold = duplicate_threshold
        self.similarity_threshold = similarity_threshold
        self._scratch: Optional[GalleryStore] = None

    def check_duplicate_face(self, new_embedding: np.ndarray, company_id: Optional[str] = None,
                             kind: Optional[str] = None) -> Tuple[bool, Optional[str]]:
        """(is_duplicate, id of the FIRST stored person with cos > threshold) - trainingServer.py:170-200.
        kind: 'employee' / 'visitor' - scan only that collection's templates of the company (an
        :class:`EnrolmentGallery` store).  The id returned is the stored `ref_id` (`doc[id_field]`,
        trainingServer.py:191) when the gallery carries one, else the row's document id."""
        store = self.store.store if isinstance(self.store, EnrolmentGallery) else self.store
        with _reading(store):            # scan + row -> id translation are one read section (compact() renumbers)
            rows, _ = self.matcher.first_above(np.asarray(new_embedding, np.float32)[None, :], self.duplicate_threshold,
                                               strict=True, company_id=enrolment_tenant(company_id, kind))
            if rows[0] < 0:
                return False, None
            pid = store.id_of(int(rows[0]))
            meta = store.metadata(pid) if pid is not None else None
        ref = (meta or {}).get("ref_id")
        return True, (ref if ref is not None else pid)

    def check_image_similarity(self, embeddings: Sequence[np.ndarray]) -> Tuple[bool, Optional[Tuple[int, int]]]:
        """(all poses show the same person, first offending pair) - trainingServer.py:202-214.  The pose
        embeddings go through the same device path: a scratch gallery of the poses, every pose matched
        against it, pairs read off in the reference's (i, j > i) order."""
        n = len(embeddings)
        if n < 2:
            return True, None
        if self._scratch is None:
            base = self.store.store if isinstance(self.store, EnrolmentGallery) else self.store
            dev = base.device if getattr(base, "device", None) is not None else base.store.device
            self._scratch = GalleryStore(dim=base.dim, capacity=16, device=dev, bf16_plane=False)
        sc = self._scratch
        if sc.rows:
            sc.remove_rows(list(range(sc.rows)))
            sc.compact()
        E = np.stack([np.asarray(e, np.float32) for e in embeddings])
        sc.append_rows(E)
        r = Matcher(sc).match(E, k=n, threshold=self.similarity_threshold, variant="scan_f32", with_ids=False)
        S = np.full((n, n), np.nan, np.float32)
        for i in range(n):
            for j in range(n):
                if r.rows[i, j] >= 0:
                    S[i, r.rows[i, j]] = r.scores[i, j]
        thr = np.float32(self.similarity_threshold)
        for i in range(n):
            for j in range(i + 1, n):
                if S[i, j] < thr:
                    return False, (i, j)
        return True, None

    def audit_duplicates(self, company_id: Optional[str] = None, kind: Optional[str] = None,
                         batch: int = 1024) -> List[Tuple[str, str, float]]:
        """:func:`find_duplicate_pairs` over this checker's gallery at its duplicate threshold (one company's
        collection with `company_id` / `kind`, as ``check_duplicate_face`` scans it)."""
        tenant = None if company_id is None and kind is None else enrolment_tenant(company_id, kind)
        return find_duplicate_pairs(self.store, self.duplicate_threshold, tenant, batch, self.matcher)

    def audit_all_duplicates(self) -> Dict[str, List[Tuple[str, str, float]]]:
        """Every company's duplicate audit in ONE pass over the gallery: {tenant key: pairs} for every tenant key the
        gallery knows (an :class:`EnrolmentGallery`: ``enrolment_tenant(company, kind)``), each value equal to
        ``audit_duplicates`` of that company and kind.  Pairs across companies are not duplicates under the
        reference's rule (trainingServer.py:170-200 scans one company's collection) and are not reported."""
        base = self.store.store if isinstance(self.store, EnrolmentGallery) else self.store
        matcher = _self_join_matcher(base, self.matcher)
        if matcher is None:
            raise ValueError("audit_all_duplicates needs a unit GalleryStore / EnrolmentGallery on this process's "
                             "matcher (raw stores and sharded galleries: audit_duplicates per company)")
        keys = base.tenant_keys()
        out: Dict[str, List[Tuple[str, str, float]]] = {key: [] for key in keys.values()}
        with _reading(base):
            tags = base.read_tags()
            for a, ia, ib, sc in _self_join_pairs(base, matcher, self.duplicate_threshold, None, True):
                key = keys.get(int(tags[a]))
                if key is not None:
                    out[key].append((ia, ib, sc))
        return out

    @staticmethod
    def template_from_poses(pose_embeddings: Sequence[np.ndarray]) -> np.ndarray:
        """trainingServer.py:355."""
        return np.mean(pose_embeddings, axis=0)


def _identity(base):
    def ident(row: int) -> Optional[str]:
        pid = base.id_of(row)
        ref = (base.metadata(pid) or {}).get("ref_id") if pid is not None else None
        return ref if ref is not None else pid
    return ident


def _self_join_matcher(base, matcher) -> Optional[Matcher]:
    """The matcher of the device self-join, or None when the store is not one it serves: a raw store, a bf16-only
    store, or a foreign matcher (a ShardedMatcher over a ShardedGallery) whose pairs need the other ranks' rows."""
    if not isinstance(base, GalleryStore) or base.bf16_only or (base.stats().flags & N.STORE_RAW):
        return None
    if matcher is None:
        return Matcher(base)
    if type(matcher) is Matcher and matcher.store is base and matcher.metric == "cosine":
        return matcher
    return None


def _self_join_pairs(base, matcher: Matcher, threshold: float, company_id: Optional[str], same_company: bool):
    """(row a, id a, id b, score) of every pair of the device self-join, strict, in the audit's order; pairs whose ids
    are equal (several templates of one person) are skipped.  The caller holds the store's read section."""
    ident = _identity(base)
    A, B, S = matcher.self_join(threshold, company_id=company_id, same_company=same_company, strict=True, max_hits=16)
    out = []
    for a, b, sc in zip(A.tolist(), B.tolist(), S.tolist()):
        ia, ib = ident(a), ident(b)
        if ia != ib:
            out.append((a, ia, ib, sc))
    return out


def find_duplicate_pairs(store, threshold: float = DUPLICATE_THRESHOLD, company_id: Optional[str] = None,
                         batch: int = 1024, matcher=None, within_companies: bool = False) -> List[Tuple[str, str, float]]:
    """Whole-gallery duplicate audit: every pair of live rows a < b (gallery order) with cos > threshold - the rule
    of the enrol-time check (trainingServer.py:170-200), applied to what is already enrolled.  company_id: only
    that tenant's rows (an :class:`EnrolmentGallery` takes the key of ``enrolment_tenant``).  within_companies: every
    company at once, each within itself (only pairs whose two rows carry the same tenant tag).  Each pair is reported
    once, from the lower row's query, as (id_a, id_b, score), ordered by row a, then score desc, then row b; pairs
    whose ids are equal are skipped (an enrolment gallery holds several templates per person: the id is the
    template's `ref_id` when it has one).
    Mechanism: a unit ``GalleryStore`` (or :class:`EnrolmentGallery`) without a foreign `matcher` runs the device
    self-join (``Matcher.self_join``: the upper triangle only, no row leaves the device).  Raw stores and sharded
    galleries with a ``ShardedMatcher`` read the rows back in batches of `batch` and send them as queries through
    ``match_range``; the scores are the same on both paths, bit for bit."""
    base = store.store if isinstance(store, EnrolmentGallery) else store
    join = _self_join_matcher(base, matcher)
    if join is not None:
        with _reading(base):
            return [(ia, ib, sc) for _, ia, ib, sc in _self_join_pairs(base, join, threshold, company_id,
                                                                         within_companies)]
    if within_companies:
        raise ValueError("within_companies runs on the device self-join only (a unit GalleryStore / "
                         "EnrolmentGallery without a foreign matcher)")
    return _find_duplicate_pairs_readback(store, threshold, company_id, batch, matcher)


def _find_duplicate_pairs_readback(store, threshold: float = DUPLICATE_THRESHOLD, company_id: Optional[str] = None,
                                   batch: int = 1024, matcher=None) -> List[Tuple[str, str, float]]:
    """The audit by readback: the stored rows are read back in batches and sent as queries through
    ``Matcher.match_range``, the pairs with rows <= a dropped on the host (every pair is computed twice).  The path
    of the stores the self-join does not serve, and the yardstick it is tested against."""
    base = store.store if isinstance(store, EnrolmentGallery) else store
    matcher = matcher if matcher is not None else Matcher(base)
    code = None if company_id is None else base.tenant_code(company_id, create=False)
    ident = _identity(base)

    pairs: List[Tuple[str, str, float]] = []
    with _reading(base):
        n = base.rows
        for r0 in range(0, n, batch):
            vecs, tags = base.read_rows(r0, min(batch, n - r0))
            live = np.nonzero((tags >= 0) if code is None else (tags == code))[0]
            if not len(live):
                continue
            res = matcher.match_range(vecs[live], threshold, company_id=company_id, max_hits=16, strict=True,
                                      with_ids=False)
            for a, rows, scores in zip((r0 + live).tolist(), res.rows, res.scores):
                later = rows > a
                if not later.any():
                    continue
                ia = ident(a)
                for b, sc in zip(rows[later].tolist(), scores[later].tolist()):
                    ib = ident(b)
                    if ia != ib:
                        pairs.append((ia, ib, sc))
    return pairs
