"""Row-sharded gallery over the GPUs of one box (SURVEY.md section 8e, BASELINE config 4).

One process per GPU (``torch.distributed``; NCCL on GPUs, gloo in the CPU tests).  Rank r holds the
contiguous block of gallery rows ``[offset_r, offset_r + n_r)``; a match is

    local fused match on every rank           (frg_match, rows returned as GLOBAL rows)
    -> exchange "p2p" (default on GPUs): frg_match_exchange - the select stage of the local match pushes each
       query's top-k into every rank's exchange buffer over NVLink peer memory the moment it is final
       (8-byte {payload, epoch} packets: the data is its own flag; torch symmetric memory supplies the peer
       pointers), and one last kernel merges every query's `world` lists as their packets arrive:
       no collective-library call on the data path
    -> exchange "nccl" (fallback; gloo in the CPU tests): ONE all-gather of the block, then the k-way merge
       kernel on every rank (frg_merge_topk_strided)

Contiguous blocks keep global row order = enrolment order, so the merge's (score desc, row asc)
order reproduces the reference's strict-'>' tie rule (infrenceServer.py:538-542) across shards.
Queries are replicated: every rank passes the same batch (``broadcast=True`` ships rank 0's).

The reference has no distributed code at all; this file is new capability, not a port.
"""
from __future__ import annotations

import ctypes as C
import functools
import threading
from typing import Callable, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _native as N
from .gallery import GalleryStore
from .matcher import LIVE_THRESHOLD, Matcher, MatchResult, RangeResult, best_first


def block_layout(F: int, k: int) -> Tuple[int, int]:
    """(bytes of the row part, bytes of one rank's packed [rows int64 | scores fp32] block).  The block is
    padded to a multiple of 8 so that every rank's row part stays int64-aligned inside the gathered buffer
    for any F*k (odd ones too)."""
    rows_bytes = F * k * 8
    return rows_bytes, rows_bytes + ((F * k * 4 + 7) & ~7)


def shard_bounds(n_rows: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous, balanced row blocks: rank r owns [lo, hi)."""
    return [((n_rows * r) // world, (n_rows * (r + 1)) // world) for r in range(world)]


def _locked(fn):
    """Id-level calls of one rank are serialised (the sync thread mutates the tables the matcher threads read):
    the reference's embeddings_lock."""
    @functools.wraps(fn)
    def wrapper(self, *a, **kw):
        with self._lock:
            return fn(self, *a, **kw)
    return wrapper


def owner_of(row: int, bounds: List[Tuple[int, int]]) -> int:
    for r, (lo, hi) in enumerate(bounds):
        if lo <= row < hi:
            return r
    return len(bounds) - 1


class ShardedGallery:
    """The local shard plus the shared view of who owns what."""

    def __init__(self, dim: int = 512, device: Optional[int] = None, group=None, store: Optional[GalleryStore] = None,
                 rank: Optional[int] = None, world: Optional[int] = None):
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self.dim = dim
        self.device = device
        self.store = store           # None in host-logic tests that inject their own local matcher
        self.bounds: List[Tuple[int, int]] = [(0, 0)] * self.world
        # the dict keys of the reference (infrenceServer.py:48-51), replicated on every rank: id <-> GLOBAL row
        self._row_of: Dict[str, int] = {}
        self._id_of: Dict[int, str] = {}
        self._meta: Dict[str, Dict] = {}
        self._tenants: Dict[str, int] = {}
        self._tenant_of: Dict[str, int] = {}     # id -> tenant code (company subset sizes without a device read)
        self._removed: set = set()   # global rows tombstoned so far
        self._anon = 0               # live rows without an id entry (synthetic fills)
        self._lock = threading.RLock()

    # ---- layout ---------------------------------------------------------------------------------
    @property
    def offset(self) -> int:
        return self.bounds[self.rank][0]

    @property
    def local_rows(self) -> int:
        lo, hi = self.bounds[self.rank]
        return hi - lo

    @property
    def total_rows(self) -> int:
        return self.bounds[-1][1]

    def plan(self, n_rows: int):
        self.bounds = shard_bounds(n_rows, self.world)
        return self.bounds[self.rank]

    @_locked
    def fill_synthetic(self, n_rows: int, seed: int = 1234):
        """Every rank materialises ITS block of the frg-synth-v1 gallery on its own GPU; row r depends
        only on (seed, r), so the data is identical at 1, 2, 4 or 8 GPUs and never touches the host."""
        lo, hi = self.plan(n_rows)
        self.store.fill_synthetic(hi - lo, lo, seed)
        self._anon = n_rows

    @_locked
    def append_local(self, vecs: np.ndarray, tags=None, prenormalised: bool = False):
        """Collective enrolment: every rank passes the SAME batch; each keeps the rows whose global
        position falls into its block after the gallery has been re-planned to the new size... which
        would move rows between ranks.  Appends therefore go to the LAST rank (global order is kept,
        blocks become unbalanced; rebalancing is a maintenance operation, DESIGN.md)."""
        n = len(vecs)
        lo, hi = self.bounds[-1]
        self.bounds = self.bounds[:-1] + [(lo, hi + n)]
        if self.rank == self.world - 1 and self.store is not None:
            self.store.append_rows(vecs, tags, prenormalised)
        return hi

    # ---- id-level API (the dict), collective: every rank makes the same calls in the same order ----
    @_locked
    def tenant_code(self, company_id: Optional[str], create: bool = True) -> int:
        """Same codes on every rank because every rank sees the same upserts in the same order."""
        if company_id is None:
            return 0
        key = str(company_id)
        if key not in self._tenants:
            if not create:
                return 0x7FFFFFFF            # a tag no row carries
            self._tenants[key] = len(self._tenants) + 1
        return self._tenants[key]

    def __len__(self):
        return len(self._row_of) + self._anon

    def __contains__(self, pid: str):
        return str(pid) in self._row_of

    def row_of(self, pid: str) -> int:
        return self._row_of.get(str(pid), -1)

    @_locked
    def id_of(self, row: int) -> Optional[str]:
        """Id of a GLOBAL row; rows filled synthetically carry the implicit id ``"%024x" % row``."""
        row = int(row)
        if row < 0:
            return None
        pid = self._id_of.get(row)
        if pid is None and row < self.total_rows and row not in self._removed:
            return "%024x" % row
        return pid

    def metadata(self, pid: str) -> Optional[Dict]:
        return self._meta.get(str(pid))

    @_locked
    def ids(self) -> List[str]:
        """Live ids in global gallery (= dict) order."""
        return [self._id_of[r] for r in sorted(self._id_of)]

    @_locked
    def count_tenant(self, company_id: Optional[str]) -> int:
        code = self.tenant_code(company_id, create=False)
        return sum(1 for c in self._tenant_of.values() if c == code)

    def stats(self):
        """Device-side figures of THIS rank's shard."""
        return self.store.stats()

    @_locked
    def load(self, ids: Sequence[str], vecs: np.ndarray, company_ids: Optional[Sequence[Optional[str]]] = None,
             meta: Optional[Sequence[Dict]] = None, prenormalised: bool = False):
        """Initial load of an EMPTY sharded gallery (the reference's load_all_embeddings,
        infrenceServer.py:260-341): the batch, in dict order, is cut into balanced contiguous blocks and each
        rank ingests only its own.  Ids must be distinct."""
        vecs = np.ascontiguousarray(vecs, dtype=np.float32).reshape(-1, self.dim)
        if self.total_rows:
            raise RuntimeError("load() needs an empty gallery; use upsert() afterwards")
        if len(ids) != len(vecs) or len(set(map(str, ids))) != len(ids):
            raise ValueError("ids must be distinct and as many as vecs")
        tags = np.array([self.tenant_code(c) for c in (company_ids or [None] * len(ids))], np.int32)
        lo, hi = self.plan(len(ids))
        if self.store is not None and hi > lo:
            self.store.append_rows(vecs[lo:hi], tags[lo:hi], prenormalised)
        for r, p in enumerate(ids):
            self._row_of[str(p)] = r
            self._id_of[r] = str(p)
            self._tenant_of[str(p)] = int(tags[r])
        if meta is not None:
            for p, m in zip(ids, meta):
                self._meta[str(p)] = m

    @_locked
    def upsert(self, ids: Sequence[str], vecs: np.ndarray, company_ids: Optional[Sequence[Optional[str]]] = None,
               meta: Optional[Sequence[Dict]] = None, prenormalised: bool = False):
        """``self.embeddings[id] = v / ||v||`` (infrenceServer.py:273,326; peopleCount.py:790,808) over the
        sharded gallery.  An existing id is overwritten in place ON ITS OWNER rank (it keeps its global
        position, as dict assignment does); new ids append at the end of the global order, i.e. to the last
        rank's block (SURVEY.md section 8e).  Position within a batch: first occurrence; content: last."""
        vecs = np.ascontiguousarray(vecs, dtype=np.float32).reshape(-1, self.dim)
        if len(ids) != len(vecs):
            raise ValueError("ids and vecs differ in length")
        if self.total_rows == 0 and len(set(map(str, ids))) == len(ids):
            return self.load(ids, vecs, company_ids, meta, prenormalised)       # the initial load: balanced blocks
        tags = np.array([self.tenant_code(c) for c in (company_ids or [None] * len(ids))], np.int32)
        last = {str(p): i for i, p in enumerate(ids)}
        new_i, old_i = [], []
        for p in dict.fromkeys(str(p) for p in ids):
            (old_i if p in self._row_of else new_i).append(last[p])
        lo, hi = self.bounds[self.rank]
        mine = [i for i in old_i if lo <= self._row_of[str(ids[i])] < hi]
        if mine and self.store is not None:
            self.store.overwrite_rows([self._row_of[str(ids[i])] - lo for i in mine], vecs[mine], tags[mine],
                                      prenormalised)
        if new_i:
            first = self.append_local(vecs[new_i], tags[new_i], prenormalised)
            for j, i in enumerate(new_i):
                self._row_of[str(ids[i])] = first + j
                self._id_of[first + j] = str(ids[i])
        for i in old_i + new_i:
            self._tenant_of[str(ids[i])] = int(tags[i])
        if meta is not None:
            for p, m in zip(ids, meta):
                self._meta[str(p)] = m

    @_locked
    def remove(self, ids: Iterable[str]) -> int:
        """``del self.embeddings[id]`` (infrenceServer.py:248-251): the owner rank tombstones the row; a later
        re-enrolment appends at the end, as ``del d[k]; d[k] = v`` does.  Unknown ids are ignored."""
        lo, hi = self.bounds[self.rank]
        gone, local = 0, []
        for p in ids:
            p = str(p)
            r = self._row_of.pop(p, None)
            if r is None:
                continue
            gone += 1
            self._id_of.pop(r, None)
            self._meta.pop(p, None)
            self._tenant_of.pop(p, None)
            self._removed.add(r)
            if lo <= r < hi:
                local.append(r - lo)
        if local and self.store is not None:
            self.store.remove_rows(local)
        return gone

    @_locked
    def remove_rows_global(self, rows: Iterable[int]) -> int:
        """Tombstone GLOBAL rows that have no id entry (synthetic fills)."""
        lo, hi = self.bounds[self.rank]
        rows = [int(r) for r in rows]
        for r in rows:
            pid = self._id_of.pop(r, None)
            if pid is not None:
                self._row_of.pop(pid, None)
                self._meta.pop(pid, None)
                self._tenant_of.pop(pid, None)
            elif r not in self._removed and self._anon > 0:
                self._anon -= 1
            self._removed.add(r)
        local = [r - lo for r in rows if lo <= r < hi]
        if local and self.store is not None:
            self.store.remove_rows(local)
        return len(rows)


class ShardedMatcher:
    def __init__(self, gallery: ShardedGallery,
                 local_match: Optional[Callable] = None, merge: Optional[Callable] = None,
                 exchange: str = "auto", metric: str = "cosine"):
        """exchange: "p2p" (the match kernels push over NVLink peer memory, a poll-only kernel merges; bounded waits), "nccl" (all-gather +
        merge kernel) or "auto" (p2p when the peer mapping can be set up, else nccl; `self.exchange` tells
        which one runs, `self.p2p_error` why not)."""
        self.g = gallery
        if metric not in N.METRICS:
            raise ValueError("metric must be one of %s" % sorted(N.METRICS))
        self.metric = metric
        self._local = local_match or self._local_cuda
        self._merge = merge or self._merge_cuda
        self._matcher = Matcher(gallery.store, metric) if gallery.store is not None else None
        self._buf = None
        if exchange not in ("auto", "p2p", "nccl"):
            raise ValueError("exchange must be auto, p2p or nccl")
        injected = local_match is not None or merge is not None      # host-logic tests: no device pieces
        self._want = "nccl" if (injected or gallery.world == 1) else exchange
        self.exchange = "nccl" if self._want == "nccl" else None      # decided at the first match
        self.p2p_error: Optional[str] = None
        self._x = None            # (tensor, handle, block_cap, slots)
        self._epoch = 0

    # ---- peer-memory exchange ---------------------------------------------------------------------
    def _p2p_setup(self, Q, F, k):
        """Collective: (re)allocates the symmetric exchange buffer for F*k slots per rank."""
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        cap, total = C.c_int64(), C.c_int64()
        N.check(N.lib.frg_exchange_bytes(self.g.world, F, k, C.byref(cap), C.byref(total)))
        group = self.g.group if self.g.group is not None else dist.group.WORLD
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")      # newer torch: enabled implicitly, the call only warns
            try:
                symm.enable_symm_mem_for_group(group.group_name)
            except Exception:        # noqa: BLE001
                pass
        t = symm.empty(int(total.value), dtype=torch.uint8, device=Q.device)
        t.zero_()                                    # flags and ticket start at 0; epochs start at 1
        hdl = symm.rendezvous(t, group)
        torch.cuda.synchronize(Q.device)
        dist.barrier(group=self.g.group)             # every buffer is zeroed before anyone pushes into it
        self._x = (t, hdl, int(cap.value), F * k)
        self._epoch = 0

    def _p2p_ready(self, Q, F, k) -> bool:
        if self._want == "nccl" or not getattr(Q, "is_cuda", False):
            return False
        if self.exchange == "nccl":
            return False
        if self._x is None or self._x[3] < F * k:
            try:
                self._p2p_setup(Q, F, k)
            except Exception as e:                   # noqa: BLE001
                self.p2p_error = repr(e)
                if self._want == "p2p":
                    raise
                self.exchange = "nccl"
                return False
        self.exchange = "p2p"
        return True

    def _match_exchange_p2p(self, Q, rows_l, scores_l, F, k, threshold, variant, tenant, out):
        """frg_match_exchange: local match whose select stage pushes each query's top-k to all ranks as it
        becomes final (the exact fallback pushes what it redoes), then the poll + merge kernel - one enqueue, no
        collective call; a void call (missing rank, other shape) is reported by check_exchange()."""
        import torch
        t, hdl, cap, _ = self._x
        rows, scores, accept = out
        self._epoch += 1
        x = N.Exchange(rank=self.g.rank, world=self.g.world, peer_bufs=int(hdl.buffer_ptrs_dev), block_cap=cap,
                       epoch=((self._epoch - 1) % 0xFFFFFFFF) + 1, flags=0)
        p = N.MatchParams(metric=N.METRICS[self.metric], variant=N.VARIANTS[variant],
                          threshold=float(np.float32(threshold)), tenant=int(tenant), row_offset=int(self.g.offset),
                          flags=0, reserved=0)
        stream = torch.cuda.current_stream(Q.device).cuda_stream
        N.check(N.lib.frg_match_exchange(
            self.g.store.handle, C.c_void_p(Q.data_ptr()), F, k, C.byref(p), C.byref(x),
            C.c_void_p(rows_l.data_ptr()), C.c_void_p(scores_l.data_ptr()), C.c_void_p(rows.data_ptr()),
            C.c_void_p(scores.data_ptr()), C.c_void_p(accept.data_ptr()), C.c_void_p(stream)))

    def check_exchange(self, clear: bool = False):
        """Host-side health check of the peer-memory exchange; call it wherever the results of earlier
        ``match`` calls are about to be trusted (it synchronises the current stream).  The poll kernel never
        hangs or traps: when a rank did not take part in a call (the ranks made different numbers of
        collective calls), passed another (F, k), or died, it gives up after FRG_EXCHANGE_TIMEOUT_MS (default
        2000), returns "no match" everywhere and leaves a status record - raised here as ``NativeError``
        (code ``ERR_STATE``) naming the call, the rank and the shapes.  After a failure the exchange buffer
        is dropped; the next ``match`` sets it up again (collective)."""
        if self._x is None:
            return
        import torch
        t = self._x[0]
        st = N.ExchangeStatus()
        stream = torch.cuda.current_stream(t.device).cuda_stream
        rc = N.lib.frg_exchange_status(t.device.index, C.c_void_p(t.data_ptr()), 1 if clear else 0,
                                       C.c_void_p(stream), C.byref(st))
        if rc != N.OK:
            self._x = None
            N.check(rc)

    def reset_exchange(self):
        """Collective: drop the exchange buffer on every rank; the next ``match`` allocates and zeroes a fresh one
        (epochs restart at 1).  The way back after ``check_exchange`` raised on ANY rank."""
        self._x = None
        self._epoch = 0

    # ---- CUDA pieces ------------------------------------------------------------------------------
    def _local_cuda(self, Q, k, threshold, variant, rows_out, scores_out, tenant=-1):
        acc = self._accept_scratch(Q)
        self._matcher.match_device(Q, k, threshold, variant=variant, row_offset=self.g.offset,
                                   out=(rows_out, scores_out, acc), tenant=tenant)

    def _accept_scratch(self, Q):
        import torch
        if self._buf is None or self._buf.shape[0] < Q.shape[0]:
            self._buf = torch.empty((Q.shape[0],), dtype=torch.uint8, device=Q.device)
        return self._buf[:Q.shape[0]]

    def _merge_cuda(self, gathered, parts, F, k, threshold, out):
        import torch
        rows, scores, accept = out
        rows_bytes, stride_bytes = block_layout(F, k)
        base = gathered.data_ptr()
        stream = torch.cuda.current_stream(gathered.device).cuda_stream
        N.check(N.lib.frg_merge_topk_strided(
            gathered.device.index, C.c_void_p(base + rows_bytes), stride_bytes // 4, C.c_void_p(base),
            stride_bytes // 8, parts, F, k, N.METRICS[self.metric], float(np.float32(threshold)),
            C.c_void_p(rows.data_ptr()), C.c_void_p(scores.data_ptr()), C.c_void_p(accept.data_ptr()),
            C.c_void_p(stream)))

    # ---- the collective match ---------------------------------------------------------------------
    def match(self, Q, k: int = 1, threshold: float = LIVE_THRESHOLD, variant: str = "auto",
              broadcast: bool = False, out=None, company_id: Optional[str] = None):
        """Q: float32 [F, dim] tensor on this rank's device, identical on every rank (or rank 0's with
        broadcast=True).  company_id: only that tenant's rows take part (infrenceServer.py:343-380).
        Returns (rows int64 [F,k] GLOBAL rows, scores fp32 [F,k], accept uint8 [F]) on every rank;
        ``ids_of(rows)`` turns rows into the reference's id strings."""
        import torch
        import torch.distributed as dist
        F = Q.shape[0]
        if broadcast and self.g.world > 1:
            dist.broadcast(Q, src=0, group=self.g.group)
        tenant = -1 if company_id is None else self.g.tenant_code(company_id, create=False)
        # packed per-rank block: F*k int64 rows, then F*k fp32 scores, padded to 8 bytes
        rows_bytes, block = block_layout(F, k)
        local = torch.empty((block,), dtype=torch.uint8, device=Q.device)
        rows_l = local[:rows_bytes].view(torch.int64).view(F, k)
        scores_l = local[rows_bytes:rows_bytes + F * k * 4].view(torch.float32).view(F, k)
        if out is None:
            out = (torch.empty((F, k), dtype=torch.int64, device=Q.device),
                   torch.empty((F, k), dtype=torch.float32, device=Q.device),
                   torch.empty((F,), dtype=torch.uint8, device=Q.device))
        if self.g.world > 1 and self._p2p_ready(Q, F, k):
            self._match_exchange_p2p(Q, rows_l, scores_l, F, k, threshold, variant, tenant, out)
            return out
        if tenant == -1:
            self._local(Q, k, threshold, variant, rows_l, scores_l)
        else:
            self._local(Q, k, threshold, variant, rows_l, scores_l, tenant=tenant)
        if self.g.world > 1:
            gathered = torch.empty((self.g.world * block,), dtype=torch.uint8, device=Q.device)
            dist.all_gather_into_tensor(gathered, local, group=self.g.group)
        else:
            gathered = local
        self._merge(gathered, self.g.world, F, k, threshold, out)
        return out

    def match_host(self, Q: np.ndarray, k: int = 1, threshold: float = LIVE_THRESHOLD,
                   company_id: Optional[str] = None, variant: str = "auto", with_ids: bool = True) -> MatchResult:
        """Host (numpy) batch in, ``MatchResult`` out - the call shape of ``Matcher.match``, so that
        ``FaceRecognitionProcessor`` / ``CameraProcessor`` run unchanged over a sharded gallery
        (``matcher=ShardedMatcher(g)``).  Collective: every rank passes the same batch."""
        import torch
        dev = torch.device("cuda", self.g.store.device if self.g.device is None else self.g.device)
        Qd = torch.from_numpy(np.ascontiguousarray(Q, dtype=np.float32).reshape(-1, self.g.dim)).to(dev)
        rows, scores, acc = self.match(Qd, k, threshold, variant, company_id=company_id)
        if self.exchange == "p2p":
            self.check_exchange()                      # results are about to be read: a void call raises here
        out = MatchResult(rows.cpu().numpy(), scores.cpu().numpy(), acc.cpu().numpy().astype(np.bool_))
        if with_ids:
            out.ids = self.ids_of(out.rows)
        return out

    def first_above(self, Q: np.ndarray, threshold: float, strict: bool = False, company_id: Optional[str] = None,
                    query_prenormalised: bool = False, local_first: Optional[Callable] = None):
        """First row IN GLOBAL GALLERY ORDER whose exact score reaches the threshold - the rule of the enrol-time
        duplicate check (trainingServer.py:170-200) over a sharded gallery: every rank scans its block
        (frg_first_match, global rows), the lowest global row over the ranks wins (one MIN all-reduce) and its
        owner's score is taken (one MAX all-reduce).  Collective.  Returns (rows int64 [F], scores fp32 [F]) as
        numpy arrays, row -1 / score -1.0 where no rank has a hit."""
        import torch
        import torch.distributed as dist
        Q = np.ascontiguousarray(Q, dtype=np.float32).reshape(-1, self.g.dim)
        tenant = -1 if company_id is None else self.g.tenant_code(company_id, create=False)
        if local_first is not None:                      # host-logic tests
            rows, scores = local_first(Q, threshold, strict, tenant)
        else:
            F = len(Q)
            rows, scores = np.empty(F, np.int64), np.empty(F, np.float32)
            p = N.MatchParams(metric=N.METRICS[self.metric], variant=N.VARIANTS["scan_f32"],
                              threshold=float(np.float32(threshold)), tenant=int(tenant),
                              row_offset=int(self.g.offset),
                              flags=(N.FIRST_STRICT if strict else 0) | (N.QUERY_PRENORMALISED if query_prenormalised else 0),
                              reserved=0)
            N.check(N.lib.frg_first_match_host(self.g.store.handle, Q.ctypes.data, F, C.byref(p),
                                               rows.ctypes.data, scores.ctypes.data))
        if self.g.world == 1:
            return rows, scores
        on_gpu = dist.get_backend(self.g.group) == "nccl"
        dev = torch.device("cuda", self.g.store.device if self.g.device is None else self.g.device) if on_gpu else "cpu"
        none = np.iinfo(np.int64).max
        r = torch.from_numpy(np.where(rows >= 0, rows, none)).to(dev)
        best = r.clone()
        dist.all_reduce(best, op=dist.ReduceOp.MIN, group=self.g.group)
        sc = torch.from_numpy(scores).to(dev)
        sc = torch.where((r == best) & (best != none), sc, torch.full_like(sc, -float("inf")))
        dist.all_reduce(sc, op=dist.ReduceOp.MAX, group=self.g.group)
        best, sc = best.cpu().numpy(), sc.cpu().numpy()
        hit = best != none
        return np.where(hit, best, -1), np.where(hit, sc, np.float32(-1.0)).astype(np.float32)

    def match_range(self, Q: np.ndarray, threshold: float, company_id: Optional[str] = None, max_hits: int = 64,
                    strict: bool = False, variant: str = "auto", with_ids: bool = True,
                    local_range: Optional[Callable] = None) -> RangeResult:
        """``Matcher.match_range`` over the row-sharded gallery.  Collective: every rank passes the same batch.
        Each rank runs the range search on its block (global rows: its row offset); ONE all-gather brings every
        rank's counts and first max_hits hits to every rank.  Ranks hold contiguous blocks, so concatenating the
        hit lists in rank order is global gallery order; the counts add up.  Queries whose total count exceeded
        max_hits are re-run once, on every rank alike (the decision is taken from the gathered counts).
        local_range(Q, threshold, strict, tenant, max_hits, row_offset) -> (counts [F], rows [F, max_hits],
        scores [F, max_hits]) replaces the device call (host-logic tests)."""
        Q = np.ascontiguousarray(Q, dtype=np.float32).reshape(-1, self.g.dim)
        tenant = -1 if company_id is None else self.g.tenant_code(company_id, create=False)
        local = local_range or (lambda Qx, thr, st, tn, mh, off: self._matcher.range_host(
            Qx, thr, tn, mh, st, variant, off))
        counts, rows, scores = self._range_gathered(Q, threshold, strict, tenant, max_hits, local)
        over = np.nonzero(counts.sum(axis=0) > max_hits)[0]
        if len(over):
            mh2 = int(counts.sum(axis=0)[over].max())
            c2, r2, s2 = self._range_gathered(Q[over], threshold, strict, tenant, mh2, local)
        lists_r, lists_s = [], []
        for f in range(len(Q)):
            j = np.searchsorted(over, f)
            if j < len(over) and over[j] == f:
                c, r, s = c2[:, j], r2[:, j], s2[:, j]
            else:
                c, r, s = counts[:, f], rows[:, f], scores[:, f]
            rr = np.concatenate([r[p, :c[p]] for p in range(len(c))])
            ss = np.concatenate([s[p, :c[p]] for p in range(len(c))])
            rr, ss = best_first(rr, ss, self.metric)
            lists_r.append(rr)
            lists_s.append(ss)
        total = np.array([len(r) for r in lists_r], np.int64)
        out = RangeResult(total, lists_r, lists_s, variant="sharded")
        if with_ids:
            out.ids = [[self.g.id_of(x) for x in r.tolist()] for r in lists_r]
        return out

    def _range_gathered(self, Q, threshold, strict, tenant, max_hits, local):
        """Every rank's (counts [world, F], rows [world, F, max_hits], scores [world, F, max_hits])."""
        F = len(Q)
        counts, rows, scores = local(Q, threshold, strict, tenant, max_hits, self.g.offset)
        if self.g.world == 1:
            return counts[None], rows[None], scores[None]
        import torch
        import torch.distributed as dist
        # one int64 block per rank: [counts F | rows F*max_hits | score bits F*max_hits]
        block = np.concatenate([np.asarray(counts, np.int64), np.asarray(rows, np.int64).ravel(),
                                np.asarray(scores, np.float32).view(np.int32).astype(np.int64).ravel()])
        on_gpu = dist.get_backend(self.g.group) == "nccl"
        dev = torch.device("cuda", self.g.store.device if self.g.device is None else self.g.device) if on_gpu else "cpu"
        mine = torch.from_numpy(block).to(dev)
        gathered = torch.empty((self.g.world * len(block),), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(gathered, mine, group=self.g.group)
        g = gathered.cpu().numpy().reshape(self.g.world, -1)
        n = F * max_hits
        return (g[:, :F], g[:, F:F + n].reshape(-1, F, max_hits),
                g[:, F + n:].astype(np.int32).view(np.float32).reshape(-1, F, max_hits))

    def ids_of(self, rows) -> List[List[Optional[str]]]:
        """Global rows of a match result -> id strings (None for unfilled slots)."""
        r = rows.cpu().numpy() if hasattr(rows, "cpu") else np.asarray(rows)
        return [[self.g.id_of(x) for x in rr] for rr in r.reshape(len(r), -1)]
