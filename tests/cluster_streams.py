"""Test infrastructure of batched unknown-face clustering (UnknownClusterer.observe_batch): face streams built to
drive every branch of the two-phase algorithm, a numpy restatement of that algorithm, and the per-face clusterer
that observe_batch must reproduce (first-match call + host mean + upsert for every face)."""
from collections import deque
from typing import List, Tuple

import numpy as np

HITS = 16                       # the pre-pass hit budget of frg_cluster_observe_host


def unit(v) -> np.ndarray:
    v = np.asarray(v, dtype=np.float64)
    return (v / np.linalg.norm(v)).astype(np.float32)


def basis(dim: int, k: int, scale: float = 1.0) -> np.ndarray:
    e = np.zeros(dim, np.float64)
    e[k] = scale
    return e


def people_stream(rng, dim: int, people: int, n: int, noise: float) -> np.ndarray:
    """n normalised faces of `people` persons in random order.  Two faces of one person score about
    1 / (1 + noise^2): noise 0.75 puts them at the 0.65 threshold."""
    centres = rng.standard_normal((people, dim))
    who = rng.integers(0, people, n)
    Q = centres[who] + noise * rng.standard_normal((n, dim))
    Q = Q / np.linalg.norm(Q, axis=1, keepdims=True)
    return Q.astype(np.float32)


def branch_streams(dim: int) -> Tuple[np.ndarray, np.ndarray]:
    """(before, batch): faces observed one at a time first, then one batch whose faces take every branch.
    Clusters 0..19 have means 0.75 e0 + 0.661 e_k (pairwise dot 0.5625 < 0.65: each founds its own cluster), so the
    probe face e0 hits all 20 (dot 0.75) - more than HITS.  A face close to cluster 20 founds it, then the batch:
      * faces 0.2 e0 + 0.98 e_k join clusters 0..15 and pull their means to 0.475 e0 + ...: a later e0 finds its 16
        listed hits touched and no longer qualifying, with a truncated list -> the rescan finds cluster 16;
      * a face whose first hit (cluster 20) a previous face of the batch joined -> recomputed, still joins;
      * an updated mean drops below the threshold for a later face that qualified against the old mean;
      * a face founds a cluster and later faces of the batch join it."""
    a, b = 0.75, float(np.sqrt(1 - 0.75 ** 2))
    before = [unit(basis(dim, 0, a) + basis(dim, k + 1, b)) for k in range(20)]
    before.append(unit(basis(dim, 30)))                                   # cluster 20: mean e30
    batch = []
    # updated mean drops below the threshold: old mean e30, q1 = 0.66 e30 + 0.751 e31, q2 = 0.66 e30 - 0.751 e31
    c, s = 0.66, float(np.sqrt(1 - 0.66 ** 2))
    batch.append(unit(basis(dim, 30, c) + basis(dim, 31, s)))            # joins 20 (touched)
    batch.append(unit(basis(dim, 30, c) - basis(dim, 31, s)))            # hit 20 in the pre-pass, not any more: founds
    batch.append(unit(basis(dim, 30, 0.9) + basis(dim, 31, 0.3)))        # first hit 20 was touched: recomputed, joins
    for k in range(16):
        batch.append(unit(basis(dim, 0, 0.2) + basis(dim, k + 1, 0.98)))  # join cluster k, mean moves off e0
    batch.append(unit(basis(dim, 0)))                                     # listed hits all touched: rescan -> 16
    batch.append(unit(basis(dim, 40)))                                    # founds a cluster in the batch
    batch.append(unit(basis(dim, 40, 0.95) + basis(dim, 41, 0.2)))       # joins the cluster founded in the batch
    batch.append(unit(basis(dim, 40, 0.9) - basis(dim, 41, 0.3)))
    return np.stack(before), np.stack(batch)


def np_mean(window) -> np.ndarray:
    return np.mean(list(window), axis=0)                                  # peopleCount.py:74


def two_phase(avg: List[np.ndarray], members: List[deque], Q: np.ndarray, threshold: float, window: int = 10,
              hits: int = HITS, dot=np.dot, stats=None):
    """Numpy restatement of the device algorithm: a pre-pass of every face against the clusters that exist before
    the batch (count + first `hits` hits in row order), then the faces in order with the touched set.  Mutates
    avg / members like a sequential clusterer; returns [(cluster, created)]."""
    thr = np.float32(threshold)
    c0 = len(avg)
    pre = [[r for r in range(c0) if dot(avg[r], q) >= thr] for q in Q]
    touched, out = set(), []
    for i, q in enumerate(Q):
        listed, count = pre[i][:hits], len(pre[i])
        cu = next((r for r in listed if r not in touched), None)
        if cu is None and count > hits:
            if stats is not None:
                stats["rescan"] = stats.get("rescan", 0) + 1
            cu = next((r for r in range(listed[-1] + 1, c0) if r not in touched and dot(avg[r], q) >= thr), None)
        if stats is not None and listed and listed[0] in touched:
            stats["first_hit_touched"] = stats.get("first_hit_touched", 0) + 1
        ct = min((r for r in touched if (cu is None or r < cu) and dot(avg[r], q) >= thr), default=None)
        dec = min((r for r in (cu, ct) if r is not None), default=None)
        if dec is None:
            d = deque(maxlen=window)
            d.append(q)
            members.append(d)
            avg.append(q)
            touched.add(len(avg) - 1)
            out.append((len(avg) - 1, True))
        else:
            if stats is not None and dec >= c0:
                stats["join_new"] = stats.get("join_new", 0) + 1
            members[dec].append(q)
            avg[dec] = np_mean(members[dec])
            touched.add(dec)
            out.append((dec, False))
    return out


class PerFaceClusterer:
    """One first-match call, a host mean and one upsert per face: the per-face path observe_batch replaces."""

    def __init__(self, dim: int = 512, threshold: float = 0.65, window: int = 10):
        import facerecognition_infrenceengine_b200 as frg
        self.store = frg.GalleryStore(dim=dim, capacity=256, bf16_plane=False, raw=True)
        self.matcher = frg.Matcher(self.store)
        self.threshold = threshold
        self.window = window
        self.members: List[deque] = []
        self.detection_count: List[int] = []

    def observe(self, face_embedding: np.ndarray) -> Tuple[int, bool]:
        q = np.ascontiguousarray(face_embedding, dtype=np.float32)
        hit = -1
        if self.members:
            rows, _ = self.matcher.first_above(q[None, :], self.threshold, strict=False, query_prenormalised=True)
            hit = int(rows[0])
        if hit >= 0:
            self.members[hit].append(q)
            avg = np.mean(list(self.members[hit]), axis=0)
            self.store.overwrite_rows([hit], avg[None, :], np.zeros(1, np.int32))
            self.detection_count[hit] += 1
            return hit, False
        d: deque = deque(maxlen=self.window)
        d.append(q)
        self.members.append(d)
        self.detection_count.append(1)
        self.store.append_rows(q[None, :], np.zeros(1, np.int32))
        return len(self.members) - 1, True

    def close(self):
        self.store.close()
