"""UnknownClusterer.observe_batch / frg_cluster_observe_host: one call per batch of unknown faces.  Every case is held
against the per-face path it replaces (tests/cluster_streams.PerFaceClusterer: one frg_first_match_host, a host
np.mean and one upsert per face): the same (cluster, created) list, the same stored means bit for bit (NaN as NaN),
the same windows and detection counts."""
import ctypes as C
from collections import deque

import numpy as np
import pytest

from cluster_streams import PerFaceClusterer, branch_streams, people_stream
from oracle import matcher_oracle as mo
from oracle import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frg():
    import facerecognition_infrenceengine_b200 as m
    return m


def same_means(a: np.ndarray, b: np.ndarray) -> bool:
    if a.shape != b.shape:
        return False
    nan_a, nan_b = np.isnan(a), np.isnan(b)
    return bool((nan_a == nan_b).all() and np.array_equal(a[~nan_a].view(np.uint32), b[~nan_b].view(np.uint32)))


def assert_same_state(uc, ref):
    assert same_means(uc.representatives(), ref.store.read_rows()[0])
    assert uc.detection_count == ref.detection_count
    assert len(uc.members) == len(ref.members)
    for d, e in zip(uc.members, ref.members):
        assert d.maxlen == e.maxlen
        assert [bytes(x) for x in d] == [bytes(x) for x in e]
    assert uc.store.stats().rows == ref.store.stats().rows == len(uc)


def run_both(frg, faces, cuts, dim=512, window=10, singles=()):
    """Observe `faces` in batches cut at `cuts` (and single observe() calls at the positions in `singles`) on one
    clusterer, face by face on the reference; compare after every call."""
    uc = frg.UnknownClusterer(dim=dim, window=window)
    ref = PerFaceClusterer(dim=dim, window=window)
    bounds = sorted(set([0, len(faces)] + list(cuts)))
    for a, b in zip(bounds[:-1], bounds[1:]):
        if a in singles and b == a + 1:
            got = [uc.observe(faces[a])]
        else:
            got = uc.observe_batch(faces[a:b])
        want = [ref.observe(q) for q in faces[a:b]]
        assert got == want
        assert_same_state(uc, ref)
    return uc, ref


def test_golden_as_one_batch(frg, golden):
    g = golden("unknown_clusters.npz")
    Q, _ = synth.queries(int(g["f"]), int(g["people"]), int(g["dim"]), seed=int(g["seed"]),
                         genuine_every=1, noise=float(g["noise"]))
    uc = frg.UnknownClusterer(dim=int(g["dim"]), campus_id="campus0")
    res = uc.observe_batch(mo.normalise_rows(Q))
    assert frg._native.last_variant() == "cluster_observe"
    assert [r[0] for r in res] == list(g["ref_cluster"])
    assert [r[1] for r in res] == list(g["ref_created"])
    assert np.array_equal(uc.representatives(), g["ref_avgs"])
    uc.close()


@pytest.mark.parametrize("seed", range(4))
def test_random_streams_in_random_batches(frg, seed):
    rng = np.random.default_rng(100 + seed)
    Q = people_stream(rng, 512, people=int(rng.integers(5, 40)), n=700, noise=float(rng.uniform(0.65, 0.85)))
    cuts = np.cumsum(rng.integers(1, 90, 40))
    cuts = [int(c) for c in cuts if c < len(Q)]
    singles = set(c for c in cuts[::3])
    cuts = sorted(set(cuts) | set(c + 1 for c in singles))
    uc, ref = run_both(frg, Q, cuts, singles=singles)
    assert max(uc.detection_count) > 10                      # windows wrapped
    assert sum(1 for n in uc.detection_count if n > 1) > 2
    uc.close()
    ref.close()


@pytest.mark.parametrize("dim", [128, 256, 512, 1024])
def test_branch_streams(frg, dim):
    before, batch = branch_streams(dim)
    uc, ref = run_both(frg, np.concatenate([before, batch]), [len(before)], dim=dim)
    got = [c for c, _ in uc.observe_batch(batch[-4:])]          # a second batch on the moved means
    assert got == [ref.observe(q)[0] for q in batch[-4:]]
    assert_same_state(uc, ref)
    uc.close()
    ref.close()


def test_small_and_degenerate_batches(frg):
    rng = np.random.default_rng(5)
    Q = people_stream(rng, 256, people=6, n=60, noise=0.7)
    Q[[3, 17, 18]] = np.nan                                       # normalised zero faces: found clusters, never match
    uc, ref = run_both(frg, Q, [1, 2, 3, 4, 20, 21], dim=256, window=4, singles={0, 1, 2, 3, 20})
    assert uc.observe_batch(np.zeros((0, 256), np.float32)) == []
    assert_same_state(uc, ref)
    uc.close()
    ref.close()


def test_window_sizes(frg):
    rng = np.random.default_rng(6)
    Q = people_stream(rng, 128, people=4, n=120, noise=0.7)
    for window in (1, 2, 16):
        uc, ref = run_both(frg, Q, [50], dim=128, window=window)
        uc.close()
        ref.close()


def test_large_batch_grows_store_and_ring(frg):
    rng = np.random.default_rng(8)
    dim = 512
    C0 = rng.standard_normal((10000, dim)).astype(np.float32)
    C0 /= np.linalg.norm(C0, axis=1, keepdims=True)
    uc = frg.UnknownClusterer(dim=dim)
    ref = PerFaceClusterer(dim=dim)
    assert all(c for _, c in uc.observe_batch(C0))              # random directions: every face founds a cluster
    ref.store.append_rows(C0, np.zeros(len(C0), np.int32))
    for q in C0:
        ref.members.append(deque([q], maxlen=10))
        ref.detection_count.append(1)
    assert_same_state(uc, ref)
    pick = rng.integers(0, len(C0), 4096)
    batch = C0[pick] + 0.6 * rng.standard_normal((4096, dim)).astype(np.float32) / np.sqrt(dim)
    batch[::3] = rng.standard_normal((len(batch[::3]), dim))
    batch /= np.linalg.norm(batch, axis=1, keepdims=True)
    batch = batch.astype(np.float32)
    got = uc.observe_batch(batch)
    want = [ref.observe(q) for q in batch]
    assert got == want
    assert_same_state(uc, ref)
    assert uc._ring[1].numel() >= len(uc)
    uc.close()
    ref.close()


def test_tombstoned_rows(frg):
    rng = np.random.default_rng(9)
    Q = people_stream(rng, 256, people=10, n=300, noise=0.7)
    uc, ref = run_both(frg, Q[:100], [40], dim=256)
    dead = [0, 3, 5]
    uc.store.remove_rows(dead)
    ref.store.remove_rows(dead)
    got = uc.observe_batch(Q[100:])
    want = [ref.observe(q) for q in Q[100:]]
    assert got == want
    assert not set(c for c, new in got if not new) & set(dead)
    assert_same_state(uc, ref)
    uc.close()
    ref.close()


def _ring(torch, cap, window, dim):
    return [torch.zeros((cap, window, dim), dtype=torch.float32, device="cuda"),
            torch.zeros(cap, dtype=torch.int32, device="cuda"), torch.zeros(cap, dtype=torch.int32, device="cuda")]


def test_tenant_through_the_c_entry_point(frg):
    """p->tenant filters which rows can be joined and tags the new ones; held against first_match + host mean."""
    import torch
    N = frg._native
    dim, window, tenant = 256, 10, 3
    rng = np.random.default_rng(10)
    Q = people_stream(rng, dim, people=8, n=200, noise=0.7)
    other = Q[:30].copy()                                           # the same people, enrolled under tag 7
    a = frg.GalleryStore(dim=dim, capacity=16, bf16_plane=False, raw=True)
    b = frg.GalleryStore(dim=dim, capacity=16, bf16_plane=False, raw=True)
    for s in (a, b):
        s.append_rows(other, np.full(len(other), 7, np.int32))       # another tenant's rows: never joined
    ring = _ring(torch, 512, window, dim)
    torch.cuda.synchronize()
    R = N.ClusterRing(ring[0].data_ptr(), ring[1].data_ptr(), ring[2].data_ptr(), 512, window)
    p = N.MatchParams(N.METRIC_COSINE, N.VARIANT_AUTO, 0.65, tenant, 0, 0, 0)
    cl, cr = np.empty(len(Q), np.int64), np.empty(len(Q), np.uint8)
    N.check(N.lib.frg_cluster_observe_host(a.handle, Q.ctypes.data, len(Q), C.byref(p), C.byref(R),
                                           cl.ctypes.data, cr.ctypes.data))
    a._rows = a.stats().rows
    wins = {}
    for i, q in enumerate(Q):
        rows, sc = np.empty(1, np.int64), np.empty(1, np.float32)
        pf = N.MatchParams(N.METRIC_COSINE, N.VARIANT_SCAN_F32, 0.65, tenant, 0, N.QUERY_PRENORMALISED, 0)
        N.check(N.lib.frg_first_match_host(b.handle, q.ctypes.data, 1, C.byref(pf), rows.ctypes.data, sc.ctypes.data))
        row = int(rows[0])
        if row >= 0:
            wins[row].append(q)
            b.overwrite_rows([row], np.mean(list(wins[row]), axis=0)[None], np.full(1, tenant, np.int32))
            assert (cl[i], cr[i]) == (row, 0)
        else:
            row = b.append_rows(q[None], np.full(1, tenant, np.int32))
            wins[row] = deque([q], maxlen=window)
            assert (cl[i], cr[i]) == (row, 1)
    va, ta = a.read_rows()
    vb, tb = b.read_rows()
    assert same_means(va, vb) and np.array_equal(ta, tb)
    assert (ta[len(other):] == tenant).all()
    a.close()
    b.close()


def test_refused_arguments_leave_the_store_unchanged(frg):
    import torch
    N = frg._native
    dim = 128
    q = np.full((4, dim), 1.0 / np.sqrt(dim), np.float32)
    cl, cr = np.empty(4, np.int64), np.empty(4, np.uint8)
    p = N.MatchParams(N.METRIC_COSINE, N.VARIANT_AUTO, 0.65, -1, 0, 0, 0)
    ring = _ring(torch, 8, 10, dim)
    torch.cuda.synchronize()

    def call(store, R, qp=q.ctypes.data, n=4):
        return N.lib.frg_cluster_observe_host(store.handle, qp, n, C.byref(p), C.byref(R), cl.ctypes.data,
                                              cr.ctypes.data)

    raw = frg.GalleryStore(dim=dim, capacity=16, bf16_plane=False, raw=True)
    raw.append_rows(q[:2], np.zeros(2, np.int32))
    before = raw.stats()
    ok = N.ClusterRing(ring[0].data_ptr(), ring[1].data_ptr(), ring[2].data_ptr(), 8, 10)
    for R, qp, n, code in [
            (N.ClusterRing(ring[0].data_ptr(), ring[1].data_ptr(), ring[2].data_ptr(), 5, 10), q.ctypes.data, 4,
             N.ERR_INVALID),                                            # capacity 5 < rows 2 + faces 4
            (N.ClusterRing(ring[0].data_ptr(), ring[1].data_ptr(), ring[2].data_ptr(), 8, 0), q.ctypes.data, 4,
             N.ERR_INVALID),
            (N.ClusterRing(ring[0].data_ptr(), ring[1].data_ptr(), ring[2].data_ptr(), 8, 17), q.ctypes.data, 4,
             N.ERR_INVALID),
            (N.ClusterRing(None, ring[1].data_ptr(), ring[2].data_ptr(), 8, 10), q.ctypes.data, 4, N.ERR_INVALID),
            (ok, None, 4, N.ERR_INVALID),
            (ok, q.ctypes.data, -1, N.ERR_INVALID)]:
        assert call(raw, R, qp, n) == code
        after = raw.stats()
        assert (after.rows, after.version, after.capacity) == (before.rows, before.version, before.capacity)
    assert same_means(raw.read_rows()[0], q[:2])
    assert call(raw, ok, q.ctypes.data, 0) == N.OK
    for kw in (dict(raw=False, bf16_plane=False), dict(raw=True, bf16_plane=True), dict(raw=False, bf16_plane=True)):
        s = frg.GalleryStore(dim=dim, capacity=16, **kw)
        assert call(s, ok) == N.ERR_UNSUPPORTED
        assert s.stats().rows == 0
        s.close()
    raw.close()


def test_first_match_after_the_call_sees_the_new_means(frg):
    rng = np.random.default_rng(11)
    Q = people_stream(rng, 512, people=5, n=80, noise=0.7)
    uc, ref = run_both(frg, Q, [], dim=512)
    probes = Q[:20] + 0.02 * rng.standard_normal((20, 512)).astype(np.float32)
    probes /= np.linalg.norm(probes, axis=1, keepdims=True)
    for thr in (0.3, 0.65):
        a = uc.matcher.first_above(probes, thr, query_prenormalised=True)
        b = ref.matcher.first_above(probes, thr, query_prenormalised=True)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    uc.close()
    ref.close()
