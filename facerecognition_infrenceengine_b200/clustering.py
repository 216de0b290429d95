"""Online clustering of unknown faces on the device (SURVEY.md section 8f-1; BASELINE config 5's
"online enrol/update").  Mirrors peopleCount.UnknownPerson (:52-91) and the matching rule of
CampusPeopleManager.process_unknown_detection (:432-500):

  * a cluster keeps its last 10 embeddings; its representative is their plain mean, NOT re-normalised
    (:63-74) -> the clusters live in a FRG_STORE_RAW gallery (rows stored as given);
  * a face is compared by RAW dot product with each representative in creation order, the running
    best is tracked, and the first cluster with dot >= 0.65 is joined (:446-452).  Every earlier
    cluster scored < 0.65, so this is "first row with dot >= 0.65": frg_first_match, one launch.
  * otherwise the face founds a new cluster (unknown_{campus}_{n+1}, :475).

The gallery is tiny and mutates at every observation.  A whole batch of faces is observed in ONE native call
(frg_cluster_observe_host, DESIGN.md section 7.7) with the result of observing them one after the other: the
windows of the clusters live on the device next to the means, in a ring the call updates.
"""
from __future__ import annotations

import ctypes as C
from collections import deque
from typing import Deque, List, Tuple

import numpy as np

from . import _native as N
from .gallery import GalleryStore
from .matcher import Matcher

UNKNOWN_SIMILARITY_THRESHOLD = 0.65     # peopleCount.py:232


class UnknownClusterer:
    def __init__(self, dim: int = 512, device: int = 0, threshold: float = UNKNOWN_SIMILARITY_THRESHOLD,
                 window: int = 10, campus_id: str = "campus"):
        self.store = GalleryStore(dim=dim, capacity=256, device=device, bf16_plane=False, raw=True)
        self.matcher = Matcher(self.store)
        self.threshold = threshold
        self.window = window
        self.campus_id = campus_id
        self.members: List[Deque[np.ndarray]] = []
        self.detection_count: List[int] = []
        self._ring = None

    def __len__(self):
        return len(self.members)

    def unknown_id(self, cluster: int) -> str:
        return "unknown_%s_%d" % (self.campus_id, cluster + 1)         # peopleCount.py:475

    def observe(self, face_embedding: np.ndarray) -> Tuple[int, bool]:
        """face_embedding: the normalised query the reference passes on (peopleCount.py:884).  Returns
        (cluster ordinal, created)."""
        return self.observe_batch(np.asarray(face_embedding)[None])[0]

    def observe_batch(self, faces: np.ndarray) -> List[Tuple[int, bool]]:
        """[observe(q) for q in faces] in one device call: the same (cluster, created) list, cluster means,
        windows and detection counts, bit for bit."""
        Q = np.ascontiguousarray(faces, dtype=np.float32).reshape(-1, self.store.dim)
        n = len(Q)
        if n == 0:
            return []
        members, lens, heads = self._ring_for(len(self.members) + n)
        ring = N.ClusterRing(members.data_ptr(), lens.data_ptr(), heads.data_ptr(), lens.numel(), self.window)
        p = N.MatchParams(N.METRIC_COSINE, N.VARIANT_AUTO, self.threshold, -1, 0, 0, 0)
        cluster, created = np.empty(n, np.int64), np.empty(n, np.uint8)
        store = self.store
        with store._lock:
            N.check(N.lib.frg_cluster_observe_host(store.handle, Q.ctypes.data, n, C.byref(p), C.byref(ring),
                                                   cluster.ctypes.data, created.ctypes.data))
            store._rows += int(created.sum())          # the new clusters were appended to the store
        out = []
        for q, c, new in zip(Q, cluster.tolist(), created.tolist()):
            if new:
                d: Deque[np.ndarray] = deque(maxlen=self.window)
                d.append(q)
                self.members.append(d)
                self.detection_count.append(1)
            else:
                self.members[c].append(q)
                self.detection_count[c] += 1
            out.append((c, bool(new)))
        return out

    def _ring_for(self, rows: int):
        """The device ring of the clusters' windows (members [cap][window][dim], len [cap], head [cap]), grown by
        doubling to hold `rows` clusters."""
        import torch
        have = 0 if self._ring is None else self._ring[1].numel()
        if have < rows:
            cap = max(have, 256)
            while cap < rows:
                cap *= 2
            dev = torch.device("cuda", self.store.device)
            ring = (torch.zeros((cap, self.window, self.store.dim), dtype=torch.float32, device=dev),
                    torch.zeros(cap, dtype=torch.int32, device=dev), torch.zeros(cap, dtype=torch.int32, device=dev))
            if self._ring is not None:
                for new, old in zip(ring, self._ring):
                    new[:have].copy_(old)
            torch.cuda.current_stream(dev).synchronize()     # the native call runs on another stream
            self._ring = ring
        return self._ring

    def representatives(self) -> np.ndarray:
        vecs, _ = self.store.read_rows()
        return vecs

    def close(self):
        self.store.close()
