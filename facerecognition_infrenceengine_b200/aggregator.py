"""Frame -> batch aggregation (SURVEY.md section 8f-4).

The reference matches one frame at a time and DROPS frames when its depth-2 queues are full
(infrenceServer.py:594-598, :629; peopleCount.py:962 processes every 2nd frame).  Here the faces of
several frames / cameras are gathered into ONE matcher call within a latency budget: below ~250
queries the match time is flat (the gallery is read once per 128 queries), so waiting a few
milliseconds for more faces is free throughput.

Host logic only (threads + futures); the matcher is injected, which also makes it testable on CPU.
"""
from __future__ import annotations

import threading
import time
from concurrent.futures import Future
from typing import Callable, List, Optional, Tuple

import numpy as np


class BatchAggregator:
    """submit(embeddings [f, dim], company_id) -> Future of (rows [f,k], scores [f,k], accept [f]).

    A batch is flushed when `max_batch` faces are waiting or the oldest request is `max_delay_ms` old.
    Requests with different company_id are batched separately (the tenant filter is per call) - unless
    `match_many_fn(Q, company_ids)` is given, a matcher with one company filter per face (``Matcher.match_tenants``):
    then one batch takes the pending requests of every company in arrival order, up to `max_batch` faces.
    Rows are positions in the gallery: if the store may be compacted while requests are in flight, let `match_fn`
    translate rows to ids itself (``Matcher.match(..., with_ids=True)`` does so inside the store's read section) or
    carry ``MatchResult.layout_version`` along (``store.ids_of(rows, layout_version=...)``).
    `workers` batches are in flight at once, each on its own host thread (= its own CUDA stream inside
    frg_match_host): with two, the copies and launch latency of one batch hide behind the kernels of the
    other (bench `e2e.concurrent`: +10 % at 1024 queries per batch, +30 % at 64)."""

    def __init__(self, match_fn: Callable[[np.ndarray, Optional[str]], Tuple[np.ndarray, np.ndarray, np.ndarray]],
                 max_batch: int = 256, max_delay_ms: float = 5.0, workers: int = 1,
                 match_many_fn: Optional[Callable[[np.ndarray, List[Optional[str]]],
                                                  Tuple[np.ndarray, np.ndarray, np.ndarray]]] = None):
        self.match_fn = match_fn
        self.match_many_fn = match_many_fn
        self.max_batch = max_batch
        self.max_delay = max_delay_ms / 1e3
        self._cv = threading.Condition()
        self._pending: List[Tuple[np.ndarray, Optional[str], Future, float]] = []
        self._stop = False
        self.batches = 0
        self.faces = 0
        self._threads = [threading.Thread(target=self._run, daemon=True) for _ in range(max(1, int(workers)))]
        for t in self._threads:
            t.start()

    def submit(self, embeddings: np.ndarray, company_id: Optional[str] = None) -> Future:
        fut: Future = Future()
        e = np.ascontiguousarray(embeddings, dtype=np.float32)
        if e.ndim != 2:
            raise ValueError("embeddings must be [faces, dim]")
        with self._cv:
            self._pending.append((e, company_id, fut, time.monotonic()))
            self._cv.notify()
        return fut

    def close(self):
        with self._cv:
            self._stop = True
            self._cv.notify_all()
        for t in self._threads:
            t.join(timeout=5)

    def _take(self):
        """Called with the lock held: the requests of the oldest request's tenant (of every tenant with
        match_many_fn), up to max_batch faces."""
        tenant = self._pending[0][1]
        take, rest, n = [], [], 0
        for item in self._pending:
            if (self.match_many_fn is not None or item[1] == tenant) and (n == 0 or n + len(item[0]) <= self.max_batch):
                take.append(item)
                n += len(item[0])
            else:
                rest.append(item)
        self._pending = rest
        return take, tenant

    def _run(self):
        while True:
            with self._cv:
                while not self._pending and not self._stop:
                    self._cv.wait()
                if self._stop and not self._pending:
                    return
                # wait for more faces, but never past the oldest request's deadline
                while not self._stop and self._pending:
                    waiting = sum(len(p[0]) for p in self._pending)
                    left = self._pending[0][3] + self.max_delay - time.monotonic()
                    if waiting >= self.max_batch or left <= 0:
                        break
                    self._cv.wait(timeout=left)
                if not self._pending:            # another worker took the batch while this one waited
                    continue
                take, tenant = self._take()
            try:
                Q = np.concatenate([t[0] for t in take], axis=0)
                if self.match_many_fn is not None:
                    rows, scores, accept = self.match_many_fn(Q, [t[1] for t in take for _ in range(len(t[0]))])
                else:
                    rows, scores, accept = self.match_fn(Q, tenant)
                with self._cv:
                    self.batches += 1
                    self.faces += len(Q)
                o = 0
                for e, _, fut, _ in take:
                    fut.set_result((rows[o:o + len(e)], scores[o:o + len(e)], accept[o:o + len(e)]))
                    o += len(e)
            except Exception as ex:          # a failed batch fails its requests, the loop goes on
                for _, _, fut, _ in take:
                    if not fut.done():
                        fut.set_exception(ex)
