"""Gallery self-join on the B200 (frg_self_join): the tensor-core path (join_tc) against the exact join scan
(join_scan), both against the range search it is defined by and against the numpy reference, the tag rules, overflow,
edge cases, refused arguments and the Python layers (Matcher.self_join, the duplicate audits)."""
import ctypes as C

import numpy as np
import pytest

from oracle import matcher_oracle as mo
from oracle import synth
from self_join_oracle import self_join_reference

pytestmark = pytest.mark.gpu

NEAR = 2e-6


@pytest.fixture(scope="module")
def frg():
    import facerecognition_infrenceengine_b200 as m
    return m


def join(frg, store, thr, row0=0, n=None, max_hits=16, variant="auto", tenant=-1, same=False, strict=False,
         flags=0, metric=0):
    """(status, counts, rows, scores, variant, launches) of one frg_self_join_host call."""
    N = frg._native
    n = store.rows - row0 if n is None else n
    c = np.full(max(n, 1), -7, np.int64)
    r = np.empty((max(n, 1), max_hits), np.int64)
    s = np.empty((max(n, 1), max_hits), np.float32)
    f = flags | (N.FIRST_STRICT if strict else 0) | (N.JOIN_SAME_TAG if same else 0)
    p = N.MatchParams(metric, N.VARIANTS[variant], float(np.float32(thr)), int(tenant), 0, f, 0)
    rc = N.lib.frg_self_join_host(store.handle, int(row0), int(n), int(max_hits), C.byref(p), c.ctypes.data,
                                  r.ctypes.data, s.ctypes.data)
    return rc, c[:n], r[:n], s[:n], N.last_variant(), N.last_launch_count()


def ok_join(frg, *a, **k):
    rc, c, r, s, v, launches = join(frg, *a, **k)
    assert rc == 0, frg._native.lib.frg_last_error()
    return c, r, s, v, launches


def same_result(x, y):
    assert np.array_equal(x[0], y[0])
    assert np.array_equal(x[1], y[1])
    assert np.array_equal(x[2].view(np.uint32), y[2].view(np.uint32))


def planted_store(frg, n, d, n_pairs, seed, plane=True, companies=1):
    """fill_synthetic rows (`companies` contiguous blocks tagged 0, 1, ...) + n_pairs planted near-copies (cos ~ 0.96;
    a copy keeps its own row's tag); returns the store and the planted pairs (a < b)."""
    store = frg.GalleryStore(dim=d, capacity=n, bf16_plane=plane)
    block = n // companies
    for t in range(companies):
        store.fill_synthetic(block, t * block, synth.GALLERY_SEED, tag=t)
    rng = np.random.default_rng(seed)
    src = rng.choice(store.rows, 2 * n_pairs, replace=False)
    A, B = src[:n_pairs], src[n_pairs:]
    vecs, t = [], []
    for a, b in zip(A.tolist(), B.tolist()):
        v, _ = store.read_rows(a, 1)
        _, tb = store.read_rows(b, 1)
        vecs.append(mo.normalise(v[0] + 0.3 * synth.gallery(1, d, b + 100)[0]))
        t.append(tb[0])
    store.overwrite_rows(B, np.stack(vecs), np.asarray(t, np.int32))
    return store, list(zip(np.minimum(A, B).tolist(), np.maximum(A, B).tolist()))


@pytest.fixture(scope="module")
def stores(frg):
    out = {d: planted_store(frg, 200_000, d, 300, d) for d in (128, 256, 512)}
    yield out
    for s, _ in out.values():
        s.close()


@pytest.mark.parametrize("d", [128, 256, 512])
def test_tc_equals_scan(frg, stores, d):
    store, pairs = stores[d]
    n = store.rows
    windows = [(1037, 5005), (n - 301, 301), (n - 1, 1)]
    if d == 512:
        windows.append((0, n))
    for thr in (0.4, 0.15):
        for row0, m in windows:
            tc = ok_join(frg, store, thr, row0, m, variant="tc_exact", strict=True)
            sc = ok_join(frg, store, thr, row0, m, variant="scan_f32", strict=True)
            assert tc[3] == "join_tc" and sc[3] == "join_scan"
            same_result(tc, sc)
            if row0 == 0 and thr == 0.4:
                got = {(a, int(b)) for a in np.nonzero(tc[0])[0].tolist() for b in tc[1][a, :tc[0][a]]}
                assert set(pairs) <= got


def test_contract_is_range_search(frg, stores):
    """Self-join row a == frg_match_range with the stored fp32 row a as the query, restricted to b > a."""
    store, _ = stores[512]
    rng = np.random.default_rng(3)
    rows = np.sort(rng.choice(store.rows, 1024, replace=False))
    c, r, s, _, _ = ok_join(frg, store, 0.4, max_hits=64, strict=True)
    G, _ = store.read_rows(0, store.rows)
    m = frg.Matcher(store)
    rc, rr, rs = m.range_host(G[rows], 0.4, -1, 256, True, "auto")
    assert rc.max() <= 256
    for i, a in enumerate(rows.tolist()):
        later = rr[i, :rc[i]] > a
        want_r, want_s = rr[i, :rc[i]][later], rs[i, :rc[i]][later]
        assert c[a] == len(want_r)
        k = min(len(want_r), 64)
        assert np.array_equal(r[a, :k], want_r[:k])
        assert np.array_equal(s[a, :k].view(np.uint32), want_s[:k].view(np.uint32))


def _small(frg, d=128, n=700, plane=True, seed=9):
    rng = np.random.default_rng(seed)
    G = synth.gallery(n, d, seed)
    for a, b in rng.choice(n, (40, 2), replace=False):
        G[b] = mo.normalise(G[a] + 0.2 * synth.gallery(1, d, int(b) + 7)[0])
    G[130] = G[3]                                   # exact copy across a tile boundary
    G[131] = G[3]
    tags = rng.integers(0, 3, n).astype(np.int32)
    tags[[3, 130, 131]] = 1
    G[200] = 0.0                                    # stored as a NaN row
    store = frg.GalleryStore(dim=d, capacity=n, bf16_plane=plane)
    store.append_rows(G, tags)
    dead = rng.choice(np.setdiff1d(np.arange(n), [3, 130, 131, 200]), 30, replace=False)
    store.remove_rows(dead)
    tags[dead] = -1
    Gs, ts = store.read_rows(0, n)
    assert np.array_equal(ts, tags)
    return store, Gs, tags


@pytest.mark.parametrize("plane", [True, False])
def test_numpy_reference(frg, plane):
    store, G, tags = _small(frg, plane=plane)
    for tenant, same in ((-1, False), (-1, True), (1, False), (2, True)):
        for thr in (0.3, 0.999):
            c, r, s, v, _ = ok_join(frg, store, thr, max_hits=64, tenant=tenant, same=same)
            assert v == ("join_tc" if plane else "join_scan")
            rc_, rr, rs = self_join_reference(G, tags, thr, tenant, same)
            S = mo.cosine_scores(G, G)
            for a in range(len(G)):
                got = dict(zip(r[a, :c[a]].tolist(), s[a, :c[a]].tolist()))
                want = dict(zip(rr[a].tolist(), rs[a].tolist()))
                near = set(np.nonzero(np.abs(S[a] - np.float32(thr)) <= NEAR)[0].tolist())
                assert set(got) - near == set(want) - near, (tenant, same, thr, a)
                for b in set(got) & set(want):
                    assert abs(got[b] - want[b]) <= max(5e-7, 2e-6 * abs(want[b]))
                assert list(r[a, :c[a]]) == sorted(got)
            if thr == 0.999 and tenant in (-1, 1):
                assert c[3] == 2 and c[130] == 1 and c[131] == 0
            assert c[200] == 0
    store.close()


def _per_tenant_loop(frg, store, thr, variant="auto", max_hits=16):
    """What FRG_JOIN_SAME_TAG must equal: row a's result from the call filtered to a's own tag."""
    _, tags = store.read_rows(0, store.rows)
    n = store.rows
    c = np.zeros(n, np.int64)
    r = np.full((n, max_hits), -1, np.int64)
    s = np.full((n, max_hits), -1.0, np.float32)
    for t in np.unique(tags[tags >= 0]).tolist():
        ct, rt, st, _, _ = ok_join(frg, store, thr, tenant=t, variant=variant, max_hits=max_hits)
        mine = tags == t
        c[mine], r[mine], s[mine] = ct[mine], rt[mine], st[mine]
    return c, r, s


def test_same_tag_layouts(frg):
    d, n = 256, 20_000
    G = synth.gallery(n, d, 21)
    rng = np.random.default_rng(4)
    for a, b in rng.choice(n, (400, 2), replace=False):
        G[b] = mo.normalise(G[a] + 0.3 * synth.gallery(1, d, int(b) + 3)[0])
    layouts = {
        "contiguous": np.repeat(np.arange(20, dtype=np.int32), n // 20),
        "interleaved": (np.arange(n) % 7).astype(np.int32),
        "stretched": np.where(np.arange(n) < n - 5, np.arange(n) // 2000, 3).astype(np.int32),
    }
    for name, tags in layouts.items():
        for variant in ("tc_exact", "scan_f32"):
            store = frg.GalleryStore(dim=d, capacity=n)
            store.append_rows(G, tags)
            want = _per_tenant_loop(frg, store, 0.4, variant)
            got = ok_join(frg, store, 0.4, same=True, variant=variant)
            same_result(got, want)
            # p->tenant together with the flag: that tenant only
            t1 = ok_join(frg, store, 0.4, tenant=3, same=True, variant=variant)
            same_result(t1, ok_join(frg, store, 0.4, tenant=3, variant=variant))
            # compaction between two calls
            store.remove_rows(rng.choice(n, 500, replace=False))
            store.compact()
            same_result(ok_join(frg, store, 0.4, same=True, variant=variant), _per_tenant_loop(frg, store, 0.4, variant))
            store.close()


def test_same_tag_device_tags(frg):
    """Tags written on the device: the store knows no extents, every tile scans to the end."""
    import torch
    N = frg._native
    d, n = 128, 6000
    G = torch.from_numpy(synth.gallery(n, d, 8)).cuda()
    G[4000] = G[10]
    tags = torch.from_numpy((np.arange(n) % 5).astype(np.int32)).cuda()
    tags[4000] = 0
    store = frg.GalleryStore(dim=d, capacity=n)
    N.check(N.lib.frg_store_upsert(store.handle, None, C.c_void_p(G.data_ptr()), C.c_void_p(tags.data_ptr()), n, 0,
                                   None))
    torch.cuda.synchronize()
    store._rows = n
    got = ok_join(frg, store, 0.4, same=True)
    same_result(got, _per_tenant_loop(frg, store, 0.4))
    assert got[0][10] == 1 and got[1][10, 0] == 4000
    store.close()


def test_truncation_and_overflow(frg):
    d = 512
    base = synth.gallery(4000, d, 31)
    G = base.copy()
    G[100:140] = base[100]                          # 39 later copies of row 100: more than max_hits
    many = np.concatenate([G, np.repeat(base[7:8], 4200, axis=0)])   # row 7 and 4200 copies: > kRangeBudget
    store = frg.GalleryStore(dim=d, capacity=len(many))
    store.append_rows(many)
    tc = ok_join(frg, store, 0.4, variant="tc_exact", max_hits=16)
    sc = ok_join(frg, store, 0.4, variant="scan_f32", max_hits=16)
    same_result(tc, sc)
    assert tc[0][7] == 4200 and tc[0][100] == 39
    A, B, S = frg.Matcher(store).self_join(0.4, max_hits=16)
    for a, cnt in ((7, 4200), (100, 39)):
        mine = A == a
        assert mine.sum() == cnt
        full = ok_join(frg, store, 0.4, row0=a, n=1, max_hits=cnt)
        assert np.array_equal(np.sort(B[mine]), full[1][0])
    store.close()


def test_edges_and_launches(frg):
    d = 256
    empty = frg.GalleryStore(dim=d, capacity=16)
    for v in ("auto", "tc_exact", "scan_f32"):
        assert join(frg, empty, 0.4, 0, 0, variant=v)[0] == 0
    assert join(frg, empty, 0.4, 0, 1)[0] == frg._native.ERR_INVALID
    empty.close()
    n = 64 * 512
    G = synth.gallery(n, d, 12)
    for variant, name in (("tc_exact", "join_tc"), ("scan_f32", "join_scan")):
        launches = []
        for tenants in (1, 64):
            store = frg.GalleryStore(dim=d, capacity=n)
            store.append_rows(G, (np.arange(n) // (n // tenants)).astype(np.int32))
            c, r, s, v, nl = ok_join(frg, store, 0.4, same=True, variant=variant)
            assert v == name
            launches.append(nl)
            one = ok_join(frg, store, 0.4, row0=n - 1, n=1, variant=variant)
            assert one[0][0] == 0 and one[1][0, 0] == -1 and one[2][0, 0] == -1.0
            assert join(frg, store, 0.4, 5, 0, variant=variant)[0] == 0
            store.close()
        assert launches[0] == launches[1]
        slabs = -(-n // frg._native.JOIN_SLAB_ROWS)
        assert launches[0] % slabs == 0


def test_refused_arguments(frg):
    N = frg._native
    d = 128
    G = synth.gallery(300, d, 2)
    plain = frg.GalleryStore(dim=d, capacity=300, bf16_plane=False)
    plain.append_rows(G)
    raw = frg.GalleryStore(dim=d, capacity=300, raw=True)
    raw.append_rows(G)
    b16 = frg.GalleryStore(dim=d, capacity=300, bf16_only=True)
    b16.append_rows(G)
    unit = frg.GalleryStore(dim=d, capacity=300)
    unit.append_rows(G)
    U, INV = N.ERR_UNSUPPORTED, N.ERR_INVALID
    assert join(frg, raw, 0.4)[0] == U
    assert join(frg, b16, 0.4)[0] == U
    assert join(frg, unit, 0.4, metric=N.METRIC_EUCLIDEAN)[0] == U
    assert join(frg, unit, 0.4, variant="tc_bf16")[0] == U
    assert join(frg, plain, 0.4, variant="tc_exact")[0] == U
    assert join(frg, unit, 0.4, flags=N.QUERY_PRENORMALISED)[0] == U
    assert join(frg, unit, 0.4, max_hits=0)[0] == INV
    assert join(frg, unit, 0.4, row0=-1, n=2)[0] == INV
    assert join(frg, unit, 0.4, row0=299, n=2)[0] == INV
    assert join(frg, unit, 0.4, flags=64)[0] == INV
    assert join(frg, plain, 0.4)[4] == "join_scan"
    for s in (plain, raw, b16, unit):
        s.close()


def test_python_layers_big(frg):
    """find_duplicate_pairs: the self-join and the readback path give the same list, order and score bits."""
    from facerecognition_infrenceengine_b200.enrol import _find_duplicate_pairs_readback
    store, pairs = planted_store(frg, 1_000_000, 512, 1000, 77)
    got = frg.find_duplicate_pairs(store, 0.4)
    want = _find_duplicate_pairs_readback(store, 0.4)
    assert got == want and len(got) >= 1000
    store.close()


def test_python_layers_enrolment(frg):
    from facerecognition_infrenceengine_b200.enrol import _find_duplicate_pairs_readback
    d = 512
    eg = frg.EnrolmentGallery(dim=d, capacity=64)
    E = synth.gallery(12, d, 77)
    E[1] = E[0]
    E[4] = E[3]
    E[9] = E[3]
    E[10] = mo.normalise(E[6] + 0.2 * synth.gallery(1, d, 5)[0])     # two globex employees
    comp = ["acme"] * 6 + ["globex"] * 6
    kinds = ["employee", "employee", "employee", "employee", "employee", "visitor"] * 2
    eg.add(["doc%d" % i for i in range(12)], E, comp, kinds,
           ref_ids=["emp0", "emp0", "emp2", "emp3", "emp4", "emp5", "g6", "g7", "g8", "g9", "g10", "g11"])
    ck = frg.EnrolmentChecker(eg)
    assert ck.audit_duplicates("acme", "employee") == _find_duplicate_pairs_readback(eg, 0.4, "acme|employee")
    assert [(a, b) for a, b, _ in ck.audit_duplicates("acme", "employee")] == [("emp3", "emp4")]
    assert ck.audit_duplicates() == _find_duplicate_pairs_readback(eg, 0.4)
    every = ck.audit_all_duplicates()
    for key in eg.store.tenant_keys().values():
        c, k = key.split("|")
        assert every[key] == ck.audit_duplicates(c, k), key
    assert every["globex|employee"] and every["acme|employee"]
    allc = frg.find_duplicate_pairs(eg, 0.4, within_companies=True)
    assert sorted(allc) == sorted(p for v in every.values() for p in v)
    eg.close()


def test_audit_all_contiguous_companies(frg):
    d, n = 512, 40_000
    store, _ = planted_store(frg, n, d, 200, 5, companies=10)
    eg = frg.EnrolmentGallery(store=store)
    for t in range(10):
        store._tenants["c%d" % t] = t          # name the tags the fill used
    ck = frg.EnrolmentChecker(eg)
    every = ck.audit_all_duplicates()
    for t in range(10):
        assert every["c%d" % t] == frg.find_duplicate_pairs(store, 0.4, company_id="c%d" % t)
    store.close()
