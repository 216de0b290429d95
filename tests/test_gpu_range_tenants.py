"""frg_match_range_tenants: one range search in which every query carries its own tenant filter.  Every result is
compared bit for bit (count, row block, score bits) with frg_match_range of that query alone with its own tenant - the
existing, oracle-pinned path."""
import ctypes as C

import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frg():
    import facerecognition_infrenceengine_b200 as m
    return m


def _params(N, tenant=-1, variant="auto", threshold=0.4, metric="cosine", strict=False, prenorm=False):
    flags = (N.FIRST_STRICT if strict else 0) | (N.QUERY_PRENORMALISED if prenorm else 0)
    return N.MatchParams(N.METRICS[metric], N.VARIANTS[variant], float(np.float32(threshold)), int(tenant), 0, flags, 0)


def tenants_call(store, Q, tenants, max_hits, **kw):
    from facerecognition_infrenceengine_b200 import _native as N
    Q = np.ascontiguousarray(Q, np.float32)
    F = len(Q)
    t = np.ascontiguousarray(tenants, np.int32)
    c, r, s = np.zeros(F, np.int64), np.empty((F, max_hits), np.int64), np.empty((F, max_hits), np.float32)
    p = _params(N, **kw)
    N.check(N.lib.frg_match_range_tenants_host(store.handle, Q.ctypes.data, F, max_hits, C.byref(p), t.ctypes.data,
                                               c.ctypes.data, r.ctypes.data, s.ctypes.data))
    return c, r, s, N.last_variant(), N.last_launch_count()


def per_query(store, Q, tenants, max_hits, **kw):
    """frg_match_range of every query alone, with its own tenant"""
    from facerecognition_infrenceengine_b200 import _native as N
    F = len(Q)
    c, r, s = np.zeros(F, np.int64), np.empty((F, max_hits), np.int64), np.empty((F, max_hits), np.float32)
    for i in range(F):
        q = np.ascontiguousarray(Q[i:i + 1], np.float32)
        p = _params(N, tenant=int(tenants[i]), **kw)
        N.check(N.lib.frg_match_range_host(store.handle, q.ctypes.data, 1, max_hits, C.byref(p), c[i:].ctypes.data,
                                           r[i:].ctypes.data, s[i:].ctypes.data))
    return c, r, s


def check(store, Q, tenants, max_hits, variant_ran=None, **kw):
    c, r, s, var, launches = tenants_call(store, Q, tenants, max_hits, **kw)
    rc, rr, rs = per_query(store, Q, tenants, max_hits, **kw)
    assert np.array_equal(c, rc)
    assert np.array_equal(r, rr)
    assert np.array_equal(s.view(np.uint32), rs.view(np.uint32))
    if variant_ran is not None:
        assert var == variant_ran
    return c, r, s, launches


# ------------------------------------------------------------------ 1 M x 512, 100 contiguous companies
N_ROWS, DIM, T = 1_000_000, 512, 10_000


@pytest.fixture(scope="module")
def big(frg):
    store = frg.GalleryStore(dim=DIM, capacity=N_ROWS)
    for t0 in range(0, N_ROWS, T):
        store.fill_synthetic(T, t0, synth.GALLERY_SEED, tag=1 + t0 // T)
    store._tenants = {"c%d" % i: i for i in range(1, N_ROWS // T + 1)}
    yield store
    store.close()


def company_queries(n_tenants, per, seed, extra_all=0, extra_unknown=0):
    """per faces of each of n_tenants companies (near a row of that company, or random), shuffled, plus extras"""
    rng = np.random.default_rng(seed)
    ten = rng.choice(np.arange(1, N_ROWS // T + 1), n_tenants, replace=False)
    tenants = np.repeat(ten, per)
    rows = (tenants - 1) * T + rng.integers(0, T, len(tenants))
    Q = synth.unit_rows(rows, DIM) + np.float32(0.03) * rng.standard_normal((len(rows), DIM)).astype(np.float32)
    Q[::3] = rng.standard_normal((len(Q[::3]), DIM)).astype(np.float32)
    Qa, _ = synth.queries(extra_all, N_ROWS, DIM) if extra_all else (np.zeros((0, DIM), np.float32), None)
    Qu = rng.standard_normal((extra_unknown, DIM)).astype(np.float32)
    Q = np.concatenate([Q, Qa, Qu]).astype(np.float32)
    tenants = np.concatenate([tenants, np.full(extra_all, -1), np.full(extra_unknown, 777)]).astype(np.int32)
    order = rng.permutation(len(Q))                      # every tenant's queries scattered through the batch
    return Q[order], tenants[order]


@pytest.mark.parametrize("n_t", [8, 64])
@pytest.mark.parametrize("per", [1, 4, 16])
def test_many_tenants_one_call(big, n_t, per):
    Q, tenants = company_queries(n_t, per, n_t * 100 + per, extra_all=5, extra_unknown=3)
    for thr in (0.4, 0.15):
        for strict in (False, True):
            c, r, s, _ = check(big, Q, tenants, 16, variant_ran="range_tc_grouped", threshold=thr, strict=strict)
            unknown = tenants == 777
            assert (c[unknown] == 0).all() and (r[unknown] == -1).all() and (s[unknown] == -1.0).all()
            if thr == 0.4:
                assert (c[tenants > 0] > 0).any()            # the near-duplicate faces find their company's rows
    # truncation: the unfiltered queries have hundreds of rows at 0.15; the first 16 in gallery order come back
    c, r, s, *_ = tenants_call(big, Q, tenants, 16, threshold=0.15)
    over = c > 16
    assert over[tenants == -1].all()
    assert (np.diff(r[over], axis=1) > 0).all()


def test_launch_count_does_not_grow_with_tenants(big):
    counts = []
    for n_t in (8, 64):
        Q, tenants = company_queries(n_t, 4, n_t)
        *_, launches = check(big, Q, tenants, 8, variant_ran="range_tc_grouped")
        counts.append(launches)
    assert counts[0] == counts[1]


def test_single_tenant_is_frg_match_range(big, frg):
    Q, _ = company_queries(1, 40, 3)
    tenants = np.full(len(Q), 5, np.int32)
    c, r, s, var, _ = tenants_call(big, Q, tenants, 16)
    m = frg.Matcher(big)
    rc, rr, rs = m.range_host(Q, 0.4, 5, 16)
    assert var == "range_tc" and frg._native.last_variant() == "range_tc"
    assert np.array_equal(c, rc) and np.array_equal(r, rr) and np.array_equal(s.view(np.uint32), rs.view(np.uint32))
    # every query "all tenants" (any negative tag): the unfiltered frg_match_range
    check(big, Q[:3], [-1, -5, -1], 4, variant_ran="range_tc")


def test_stretched_company_and_overflow(frg):
    """a company re-enrolled once at the gallery's end (tile list), and a company whose rows hold thousands of
    near-duplicates of its queries (more candidates than the filter keeps per query -> the exact scan with the query's
    own tenant), in one call with companies that do not overflow"""
    n = 300_000
    store = frg.GalleryStore(dim=DIM, capacity=n + 8192)
    for t0 in range(0, n, T):
        store.fill_synthetic(T, t0, synth.GALLERY_SEED, tag=1 + t0 // T)
    rng = np.random.default_rng(5)
    store.overwrite_rows([n - 1], synth.unit_rows([n - 1], DIM), np.array([7], np.int32), prenormalised=True)
    base = synth.unit_rows([3 * T + 17], DIM)[0]
    dups = base[None, :] + np.float32(1e-2) * rng.standard_normal((6000, DIM)).astype(np.float32)
    store.append_rows(dups, np.full(6000, 4, np.int32))          # tenant 4: its block + 6000 near-duplicates
    Qs, ts = [], []
    for t in (7, 4, 9, 12, -1):
        rows = (abs(t) - 1) * T + rng.integers(0, T, 6) if t > 0 else rng.integers(0, n, 6)
        Qs.append(synth.unit_rows(rows, DIM) + np.float32(0.02) * rng.standard_normal((6, DIM)).astype(np.float32))
        ts += [t] * 6
    Qs.append(np.repeat(base[None, :], 4, 0) + np.float32(1e-2) * rng.standard_normal((4, DIM)).astype(np.float32))
    ts += [4] * 4
    Q = np.concatenate(Qs).astype(np.float32)
    tq = np.array(ts, np.int32)
    perm = rng.permutation(len(Q))
    for max_hits in (1, 16):
        c, r, s, _ = check(store, Q[perm], tq[perm], max_hits, variant_ran="range_tc_grouped")
        assert (c[perm >= len(Q) - 4] > 4096).all()                 # overflowed: redone by the exact scan
        assert (c[tq[perm] == 7] > 0).all()
    store.close()


# ------------------------------------------------------------------ the exact path
def test_exact_path_stores(frg):
    rng = np.random.default_rng(9)
    n = 20_000
    G = rng.standard_normal((n, 128)).astype(np.float32)
    tags = (np.arange(n) // 5000 + 1).astype(np.int32)
    Q = G[rng.integers(0, n, 24)] + np.float32(0.05) * rng.standard_normal((24, 128)).astype(np.float32)
    tq = np.array([1, 2, 3, 4, -1, 8] * 4, np.int32)
    stores = {
        "plain": frg.GalleryStore(dim=128, capacity=n),
        "raw": frg.GalleryStore(dim=128, capacity=n, raw=True),
        "no_plane": frg.GalleryStore(dim=128, capacity=n, bf16_plane=False),
    }
    for s in stores.values():
        s.append_rows(G, tags)
    for thr, strict in ((0.2, False), (0.3, True)):
        check(stores["plain"], Q, tq, 8, variant="scan_f32", variant_ran="range_scan_tenants", threshold=thr,
              strict=strict)
        check(stores["no_plane"], Q, tq, 8, variant_ran="range_scan_tenants", threshold=thr, strict=strict)
    Qn = Q / np.linalg.norm(Q, axis=1, keepdims=True)
    check(stores["plain"], Qn, tq, 8, variant_ran="range_scan_tenants", threshold=0.2, prenorm=True)
    Qr = G[:24] * 1.1 + 0.05
    c, *_ = check(stores["raw"], Qr, tq, 64, variant_ran="range_scan_tenants", metric="euclidean", threshold=14.0)
    assert c.max() > 0
    check(stores["raw"], Qr, tq, 4, variant_ran="range_scan_tenants", metric="euclidean", threshold=14.0,
          strict=True)
    for s in stores.values():
        s.close()


# ------------------------------------------------------------------ store states
def test_store_states(frg):
    """tiny and interleaved companies, tombstones, NaN rows, zero queries, compaction between two calls, nq = 0"""
    rng = np.random.default_rng(11)
    n = 40_000
    for bf16_plane in (True, False):
        store = frg.GalleryStore(dim=256, capacity=n + 4096, bf16_plane=bf16_plane)
        variant = "range_tc_grouped" if bf16_plane else "range_scan_tenants"
        G = rng.standard_normal((n, 256)).astype(np.float32)
        tags = np.where(np.arange(n) < 20_000, np.arange(n) % 3 + 1, 10 + (np.arange(n) - 20_000) // 100).astype(np.int32)
        store.append_rows(G, tags)
        store.append_rows(np.full((1, 256), np.nan, np.float32), np.array([12], np.int32))
        store.remove_rows(rng.integers(0, n, 500))
        tq = np.array([1, 2, 3, 10, 11, 150, 209, -1, 999, 12] * 6, np.int32)
        rows = np.array([np.nonzero(tags == t)[0][i % 50] if t in tags else 0 for i, t in enumerate(tq)])
        Q = G[rows] + np.float32(0.1) * rng.standard_normal((len(tq), 256)).astype(np.float32)
        Q[5] = 0
        for max_hits in (1, 8):
            check(store, Q, tq, max_hits, variant_ran=variant, threshold=0.3)
            check(store, Q, tq, max_hits, variant_ran=variant, threshold=0.05, strict=True)
        c, *_ = tenants_call(store, Q[:0], tq[:0], 3)
        assert c.shape == (0,)
        check(store, Q[:1], tq[:1], 3)
        store.compact()
        check(store, Q, tq, 5, variant_ran=variant, threshold=0.3)
        store.close()


def test_device_written_tags_and_empty_gallery(frg):
    """tags upserted from device arrays (the store's tenant extents become unknown: every tile, every row's tag
    tested); an empty gallery gives counts 0 and "none" slots"""
    import torch
    from facerecognition_infrenceengine_b200 import _native as N
    store = frg.GalleryStore(dim=128, capacity=8192)
    Q = np.random.default_rng(2).standard_normal((20, 128)).astype(np.float32)
    t = np.array([1, 2, -1, 3] * 5, np.int32)
    c, r, s, _ = check(store, Q, t, 3)
    assert (c == 0).all() and (r == -1).all() and (s == -1.0).all()
    rng = np.random.default_rng(3)
    G = torch.from_numpy(rng.standard_normal((6000, 128)).astype(np.float32)).cuda()
    tags = torch.from_numpy((np.arange(6000) // 2000 + 1).astype(np.int32)).cuda()
    N.check(N.lib.frg_store_upsert(store.handle, None, C.c_void_p(G.data_ptr()), C.c_void_p(tags.data_ptr()), 6000,
                                   0, None))
    torch.cuda.synchronize()
    Q = G[::300].cpu().numpy() + np.float32(0.05)
    tq = (np.arange(len(Q)) % 4).astype(np.int32)
    check(store, Q, tq, 5, variant_ran="range_tc_grouped", threshold=0.2)
    check(store, Q, tq, 5, variant_ran="range_scan_tenants", variant="scan_f32", threshold=0.2)
    store.close()


# ------------------------------------------------------------------ arguments
def test_arguments(frg):
    from facerecognition_infrenceengine_b200 import _native as N
    d = 128
    unit = frg.GalleryStore(dim=d, capacity=64)
    unit.append_rows(np.eye(8, d, dtype=np.float32), np.arange(8, dtype=np.int32) % 2 + 1)
    bf = frg.GalleryStore(dim=d, capacity=64, bf16_only=True)
    bf.append_rows(np.eye(8, d, dtype=np.float32))
    q = np.ascontiguousarray(np.eye(2, d, dtype=np.float32))
    t = np.array([1, 2], np.int32)
    c, r, s = np.zeros(2, np.int64), np.zeros(8, np.int64), np.zeros(8, np.float32)

    def both(store, max_hits=4, tenants=t, Qp=q, **kw):
        """(status of frg_match_range_tenants_host, of frg_match_range_tenants, of frg_match_range_host)"""
        p = _params(N, **kw)
        tp = None if tenants is None else tenants.ctypes.data
        host = N.lib.frg_match_range_tenants_host(store.handle, Qp.ctypes.data, 2, max_hits, C.byref(p), tp,
                                                  c.ctypes.data, r.ctypes.data, s.ctypes.data)
        p1 = _params(N, tenant=1, **kw)
        single = N.lib.frg_match_range_host(store.handle, Qp.ctypes.data, 2, max_hits, C.byref(p1), c.ctypes.data,
                                            r.ctypes.data, s.ctypes.data)
        return host, single

    def device(store, max_hits=4, tenants=t, **kw):
        import torch
        p = _params(N, **kw)
        Qd = torch.from_numpy(q).cuda()
        cd = torch.zeros(2, dtype=torch.int64, device="cuda")
        rd = torch.zeros((2, max(max_hits, 1)), dtype=torch.int64, device="cuda")
        sd = torch.zeros((2, max(max_hits, 1)), dtype=torch.float32, device="cuda")
        tp = None if tenants is None else tenants.ctypes.data
        rc = N.lib.frg_match_range_tenants(store.handle, C.c_void_p(Qd.data_ptr()), 2, max_hits, C.byref(p), tp,
                                           C.c_void_p(cd.data_ptr()), C.c_void_p(rd.data_ptr()),
                                           C.c_void_p(sd.data_ptr()), None)
        torch.cuda.synchronize()
        return rc

    cases = [
        (unit, dict(max_hits=0), N.ERR_INVALID),
        (unit, dict(variant="tc_bf16"), N.ERR_UNSUPPORTED),
        (bf, dict(), N.ERR_UNSUPPORTED),
        (unit, dict(variant="tc_exact", metric="euclidean"), N.ERR_UNSUPPORTED),
    ]
    for store, kw, want in cases:
        host, single = both(store, **kw)
        assert host == single == want, kw
        assert device(store, **kw) == want, kw
    host, _ = both(unit, tenants=None)
    assert host == N.ERR_INVALID and device(unit, tenants=None) == N.ERR_INVALID
    # nq = 0 with no tenants is fine
    p = _params(N)
    assert N.lib.frg_match_range_tenants_host(unit.handle, None, 0, 4, C.byref(p), None, None, None, None) == N.OK
    # host and device entry points agree
    import torch
    Qd = torch.from_numpy(q).cuda()
    cd = torch.zeros(2, dtype=torch.int64, device="cuda")
    rd = torch.zeros((2, 4), dtype=torch.int64, device="cuda")
    sd = torch.zeros((2, 4), dtype=torch.float32, device="cuda")
    p = _params(N, threshold=0.5)
    N.check(N.lib.frg_match_range_tenants(unit.handle, C.c_void_p(Qd.data_ptr()), 2, 4, C.byref(p), t.ctypes.data,
                                          C.c_void_p(cd.data_ptr()), C.c_void_p(rd.data_ptr()),
                                          C.c_void_p(sd.data_ptr()), None))
    torch.cuda.synchronize()
    hc, hr, hs, *_ = tenants_call(unit, q, t, 4, threshold=0.5)
    assert np.array_equal(cd.cpu().numpy(), hc) and np.array_equal(rd.cpu().numpy(), hr)
    assert np.array_equal(sd.cpu().numpy().view(np.uint32), hs.view(np.uint32))
    assert list(hc) == [1, 1] and list(hr[:, 0]) == [0, 1]         # row 0 carries tag 1, row 1 tag 2
    for st in (unit, bf):
        st.close()


# ------------------------------------------------------------------ Python
def test_python_layers(frg):
    rng = np.random.default_rng(4)
    n = 30_000
    store = frg.GalleryStore(dim=512, capacity=n)
    ids = ["p%d" % i for i in range(n)]
    comp = ["acme" if i < 10_000 else ("globex" if i < 20_000 else "initech") for i in range(n)]
    G = rng.standard_normal((n, 512)).astype(np.float32)
    store.upsert(ids, G, comp)
    m = frg.Matcher(store)
    pick = rng.integers(0, n, 40)
    Q = G[pick] + np.float32(0.05) * rng.standard_normal((40, 512)).astype(np.float32)
    Q[:4] = G[:4]                                          # an unfiltered query with many hits at a low threshold
    cids = [comp[p] if i % 4 else ("globex" if i % 8 == 0 else None) for i, p in enumerate(pick)]
    cids[3] = "nobody"
    for thr, max_hits in ((0.4, 64), (0.12, 2)):
        res = m.match_range_tenants(Q, cids, thr, max_hits=max_hits)
        assert res.variant == "range_tc_grouped"
        if max_hits == 2:
            assert (res.counts > 2).any()                  # the retry of the queries over max_hits ran
        for i in range(len(Q)):
            one = m.match_range(Q[i:i + 1], thr, company_id=cids[i], max_hits=max_hits)
            assert res.counts[i] == one.counts[0]
            assert np.array_equal(res.rows[i], one.rows[0])
            assert np.array_equal(res.scores[i].view(np.uint32), one.scores[0].view(np.uint32))
            assert res.ids[i] == one.ids[0]
        assert res.counts[3] == 0 and res.ids[3] == []
    store.close()


@pytest.mark.parametrize("plane", [False, True])
def test_check_duplicate_faces(frg, plane):
    from facerecognition_infrenceengine_b200.enrol import EnrolmentChecker, EnrolmentGallery
    from facerecognition_infrenceengine_b200.sharded import ShardedGallery, ShardedMatcher
    rng = np.random.default_rng(7)
    n, d = 6000, 512
    eg = EnrolmentGallery(store=frg.GalleryStore(dim=d, capacity=n, bf16_plane=plane))
    G = rng.standard_normal((n, d)).astype(np.float32)
    companies = ["co%d" % (i // 500) for i in range(n)]
    kinds = ["employee" if i % 3 else "visitor" for i in range(n)]
    refs = ["ref%d" % (i // 2) if i % 5 else None for i in range(n)]
    eg.add(["doc%d" % i for i in range(n)], G, companies, kinds, refs)
    chk = EnrolmentChecker(eg)
    pick = rng.integers(0, n, 48)
    E = G[pick] + np.float32(0.3) * rng.standard_normal((48, d)).astype(np.float32)
    E[::5] = rng.standard_normal((len(E[::5]), d)).astype(np.float32)        # new people
    cids = [companies[p] if i % 7 else "co%d" % ((pick[i] // 500 + 1) % 12) for i, p in enumerate(pick)]
    cids[2] = "nobody"                                                      # a company with no rows
    cids[9] = None
    ks = [kinds[p] if i % 4 else ("visitor" if kinds[p] == "employee" else "employee") for i, p in enumerate(pick)]
    ks[11] = None
    got = chk.check_duplicate_faces(E, cids, ks)
    want = [chk.check_duplicate_face(E[i], cids[i], ks[i]) for i in range(len(E))]
    assert got == want
    assert any(g[0] for g in got) and not all(g[0] for g in got)
    assert chk.check_duplicate_faces(E[:6], cids[:6]) == [chk.check_duplicate_face(E[i], cids[i]) for i in range(6)]
    assert chk.check_duplicate_faces(E[:0], []) == []
    g = ShardedGallery(dim=d, store=eg.store, rank=0, world=1)
    g.plan(n)
    with pytest.raises(NotImplementedError):
        EnrolmentChecker(g, matcher=ShardedMatcher(g)).check_duplicate_faces(E[:2], cids[:2])
    eg.close()
