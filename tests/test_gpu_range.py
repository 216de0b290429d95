"""Range search on the B200: the tensor-core path (range_tc) against the exact counting scan (range_scan), both against
the numpy reference, the special cases it must reduce to (first_match, top-k), masks and windows, the Python layers
and the whole-gallery duplicate audit."""
import numpy as np
import pytest

from oracle import matcher_oracle as mo
from oracle import synth
from range_oracle import range_search

pytestmark = pytest.mark.gpu

NEAR = 2e-6          # rows whose reference score lies this close to the threshold may fall either way
STOL = 5e-7


@pytest.fixture(scope="module")
def frg():
    import facerecognition_infrenceengine_b200 as m
    return m


def raw_range(frg, store, Q, thr, max_hits, variant, tenant=-1, strict=False, metric="cosine"):
    m = frg.Matcher(store, metric=metric)
    c, r, s = m.range_host(Q, thr, tenant, max_hits, strict, variant)
    return c, r, s, frg._native.last_variant()


def same_raw(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


def check_against_reference(c, rows, scores, Q, G, thr, mask=None, strict=False, metric="cosine"):
    """c / rows / scores: a COMPLETE gallery-order result ([F, >= max count])."""
    ref_c, ref_r, ref_s = range_search(Q, G, thr, mask=mask, strict=strict, metric=metric)
    S = mo.cosine_scores(Q, G) if metric == "cosine" else None
    for f in range(len(Q)):
        got = {int(r): float(s) for r, s in zip(rows[f, :c[f]], scores[f, :c[f]])}
        want = dict(zip(ref_r[f].tolist(), ref_s[f].tolist()))
        if metric == "cosine":
            near = set(np.nonzero(np.abs(S[f] - np.float32(thr)) <= NEAR)[0].tolist())
        else:
            near = {r for r in set(got) | set(want) if abs((got.get(r, want.get(r))) - thr) <= NEAR}
        assert set(got) - near == set(want) - near, f
        assert c[f] - len(set(got) & near) == ref_c[f] - len(set(want) & near), f
        for r in set(got) & set(want):
            # fp32 sums of 128-512 products: the rounding grows with the score (a self-match sits 1e-6 from 1.0)
            tol = max(STOL, 2e-6 * abs(want[r])) if metric == "cosine" else 1e-5
            assert abs(got[r] - want[r]) <= tol, (f, r)
        assert list(rows[f, :c[f]]) == sorted(got), f                      # gallery order


@pytest.fixture(scope="module")
def big(frg):
    n, d = 1_000_000, 512
    store = frg.GalleryStore(dim=d, capacity=n)
    store.fill_synthetic(n, 0, synth.GALLERY_SEED)
    Q, _ = synth.queries(1024, n, d)
    yield store, Q
    store.close()


@pytest.mark.parametrize("thr", [0.4, 0.15])
def test_tc_equals_scan_1m(frg, big, thr):
    """1 M x 512, all 1024 benchmark queries (CTA-pair filter) and the first 100 (single-CTA): identical counts, rows
    and scores.  0.15 is ~3.4 sigma of a random pair at dim 512: ~300 hits per query, so max_hits = 16 truncates."""
    store, Q = big
    for F in (1024, 100):
        tc = raw_range(frg, store, Q[:F], thr, 16, "tc_exact")
        ex = raw_range(frg, store, Q[:F], thr, 16, "scan_f32")
        assert tc[3] == "range_tc" and ex[3] == "range_scan"
        same_raw(tc, ex)
        au = raw_range(frg, store, Q[:F], thr, 16, "auto")
        assert au[3] == "range_tc"
        same_raw(tc, au)
        if thr == 0.15:
            assert (tc[0] > 16).mean() > 0.9 and (tc[1][tc[0] >= 16] >= 0).all()
        assert (tc[1][:, 1:] > tc[1][:, :-1])[tc[1][:, 1:] >= 0].all()            # rows ascending


@pytest.mark.parametrize("d,thr", [(128, 0.3), (256, 0.21), (512, 0.15)])
def test_dims_against_reference(frg, d, thr):
    n = 120_000
    G = synth.gallery(n, d, 7)
    store = frg.GalleryStore(dim=d, capacity=n)
    store.append_rows(G, prenormalised=True)
    Q, _ = synth.queries(200, n, d, seed=3, gallery_seed=7)
    for F in (60, 200):
        tc = raw_range(frg, store, Q[:F], thr, 1024, "tc_exact")
        ex = raw_range(frg, store, Q[:F], thr, 1024, "scan_f32")
        same_raw(tc, ex)
        assert tc[0].max() <= 1024 and tc[0].sum() > F
        check_against_reference(tc[0], tc[1], tc[2], Q[:F], G, thr)
    store.close()


def test_first_match_and_topk_are_special_cases(frg):
    n, d = 50_000, 512
    G = synth.gallery(n, d, 9)
    tags = np.where(np.arange(n) < 20_000, 1, 2).astype(np.int32)
    G[30_000:30_010] = G[25_000]
    store = frg.GalleryStore(dim=d, capacity=n)
    store.append_rows(G, tags, prenormalised=True)
    Q = np.concatenate([G[[25_000, 100, 40_000]], synth.queries(60, n, d, seed=1, gallery_seed=9)[0]])
    m = frg.Matcher(store)
    for thr in (0.4, 0.16):
        for tenant in (-1, 1, 2):
            c, r, s = m.range_host(Q, thr, tenant, 1, True, "auto")
            # first_above takes company ids; tenant codes are given straight to the native call here
            p = frg.matcher._params("cosine", "scan_f32", thr, tenant, 0)
            p.flags = frg._native.FIRST_STRICT
            fr, fs = np.empty(len(Q), np.int64), np.empty(len(Q), np.float32)
            import ctypes as C
            frg._native.check(frg._native.lib.frg_first_match_host(store.handle, Q.ctypes.data, len(Q), C.byref(p),
                                                                    fr.ctypes.data, fs.ctypes.data))
            assert np.array_equal(r[:, 0], fr) and np.array_equal(s[:, 0], fs), (thr, tenant)
            assert ((c > 0) == (fr >= 0)).all()
    # top-k: when count <= k the complete best-first list is match()'s accepted prefix
    for k in (1, 5, 16):
        res = m.match_range(Q, 0.16, max_hits=2, with_ids=False)
        top = m.match(Q, k, 0.16, with_ids=False)
        for f in range(len(Q)):
            if res.counts[f] <= k:
                acc = top.scores[f] >= np.float32(0.16)
                assert np.array_equal(res.rows[f], top.rows[f][acc]) and np.array_equal(res.scores[f], top.scores[f][acc])
    store.close()


def test_overflow_and_degenerate_galleries_fall_back(frg):
    d, n = 512, 60000
    G = synth.gallery(n, d, 31)
    dup = np.arange(1000, 9000, 2)                          # 4000 copies of row 7
    G[dup] = G[7]
    store = frg.GalleryStore(dim=d, capacity=n)
    store.append_rows(G, prenormalised=True)
    Q, _ = synth.queries(6, n, d, seed=8, gallery_seed=31)
    Q[2] = G[7] + 0.001
    Q[4] = G[7]
    for mh in (1, 64, 8192):
        tc = raw_range(frg, store, Q, 0.4, mh, "tc_exact")
        ex = raw_range(frg, store, Q, 0.4, mh, "scan_f32")
        same_raw(tc, ex)
        want = sorted([7] + list(dup))
        assert tc[0][4] == 4001 and tc[0][2] == 4001
        assert list(tc[1][4, :min(mh, 4001)]) == want[:mh]
    check_against_reference(tc[0], tc[1], tc[2], Q, G, 0.4)
    store.close()
    # the same template 50 000 times: every segment of every CTA overflows; F > 128 for the pair kernels
    n = 50_000
    g = synth.gallery(1, d, 5)[0]
    store = frg.GalleryStore(dim=d, capacity=n)
    store.append_rows(np.repeat(g[None], n, axis=0), prenormalised=True)
    other = synth.gallery(1, d, 6)[0]
    Q = np.concatenate([np.stack([g, other]), np.repeat(g[None], 140, axis=0)])
    tc = raw_range(frg, store, Q, 0.4, 100, "tc_exact")
    same_raw(tc, raw_range(frg, store, Q, 0.4, 100, "scan_f32"))
    assert tc[0][0] == n and tc[0][1] == 0 and (tc[0][2:] == n).all()
    assert (tc[1][0] == np.arange(100)).all() and (tc[1][1] == -1).all() and (tc[2][1] == -1.0).all()
    store.close()


@pytest.mark.parametrize("copies", [1, 200])
def test_row_just_above_threshold_survives_the_bf16_filter(frg, copies):
    """tests/rounding_case.py row A: its bf16 score sits below the exact one by nearly eps; a threshold just under
    the exact score must still return it (the floor is threshold - eps[q])."""
    from rounding_case import adversarial_pair
    rng = np.random.default_rng(2)
    n, d = 4094, 512
    G = mo.normalise_rows(rng.standard_normal((n, d)).astype(np.float32))
    A, B, q = adversarial_pair(0)
    G = np.concatenate([G[:1000], B[None], G[1000:3000], A[None], G[3000:]])
    rowA = 3001
    store = frg.GalleryStore(dim=d, capacity=len(G))
    store.append_rows(G, prenormalised=True)
    Q = np.concatenate([np.repeat(q[None], copies, axis=0), rng.standard_normal((5, d)).astype(np.float32)])
    exact = raw_range(frg, store, Q[:1], -2.0, len(G), "scan_f32")
    sA = exact[2][0, rowA]
    thr = float(np.nextafter(sA, np.float32(-1)))
    tc = raw_range(frg, store, Q, thr, 16, "tc_exact")
    same_raw(tc, raw_range(frg, store, Q, thr, 16, "scan_f32"))
    assert (tc[1][:copies] == rowA).any(axis=1).all()
    store.close()


def test_tenants_tombstones_nan_and_compaction(frg):
    d = 256
    n = 100_000
    G = synth.gallery(n, d, 17)
    tags = np.full(n, 3, np.int32)
    tags[:10_000] = 1                                  # a contiguous company block
    tags[50_000:60_000:2] = 2                          # an interleaved company
    tags[99_999] = 1                                   # one re-enrolment at the far end: company 1 is stretched
    G[[10, 20_000, 70_000]] = 0                        # zero rows: NaN after normalisation, never match
    store = frg.GalleryStore(dim=d, capacity=n)
    ids = ["p%d" % i for i in range(n)]
    store.upsert(ids, G, ["c%d" % t for t in tags])
    Gn, _ = store.read_rows(0, n)                      # the rows as the device normalised them
    Q = np.concatenate([Gn[[5, 50_000, 99_999, 30]], np.zeros((1, d), np.float32),
                        synth.queries(40, n, d, seed=2, gallery_seed=17)[0]])
    removed = np.arange(3, n, 97)
    store.remove([ids[i] for i in removed])
    live = np.ones(n, bool)
    live[removed] = False
    G_now, tags_now = Gn, tags
    for _ in range(2):
        for company, code in ((None, None), ("c1", 1), ("c2", 2), ("c3", 3)):
            tenant = -1 if company is None else store.tenant_code(company, create=False)
            mask = live if code is None else live & (tags_now == code)
            for thr in (0.22, -2.0):
                tc = raw_range(frg, store, Q, thr, 5000, "tc_exact", tenant)
                same_raw(tc, raw_range(frg, store, Q, thr, 5000, "scan_f32", tenant))
                if thr > -1:
                    check_against_reference(tc[0], tc[1], tc[2], Q, G_now, thr, mask=mask)
                else:
                    want = np.nonzero(mask & ~np.isnan(G_now).any(axis=1))[0]
                    assert (tc[0][:4] == len(want)).all() and tc[0][4] == 0            # zero query: no hits
                    m = min(5000, len(want))
                    assert (tc[1][:4, :m] == want[:m]).all()
        # compaction renumbers rows: the results follow the new layout
        store.compact()
        G_now, tags_now = G_now[live], tags_now[live]
        live = np.ones(len(G_now), bool)
    store.close()


def test_arguments_and_euclidean(frg):
    from facerecognition_infrenceengine_b200 import _native as N
    d = 128
    unit = frg.GalleryStore(dim=d, capacity=64)
    unit.append_rows(np.eye(8, d, dtype=np.float32))
    q = np.eye(2, d, dtype=np.float32)
    m = frg.Matcher(unit)

    def code(fn):
        with pytest.raises(frg.NativeError) as e:
            fn()
        return e.value.code
    assert code(lambda: m.range_host(q, 0.5, -1, 0)) == N.ERR_INVALID
    p = frg.matcher._params("cosine", "auto", 0.5, -1, 0)
    p.metric = 7
    import ctypes as C
    c, r, s = np.zeros(2, np.int64), np.zeros(2, np.int64), np.zeros(2, np.float32)
    assert N.lib.frg_match_range_host(unit.handle, q.ctypes.data, 2, 1, C.byref(p), c.ctypes.data, r.ctypes.data,
                                      s.ctypes.data) == N.ERR_INVALID
    assert N.lib.frg_match_range_host(unit.handle, None, 2, 1, C.byref(frg.matcher._params("cosine", "auto", 0.5, -1, 0)),
                                      c.ctypes.data, r.ctypes.data, s.ctypes.data) == N.ERR_INVALID
    assert code(lambda: m.range_host(q, 0.5, -1, 4, variant="tc_bf16")) == N.ERR_UNSUPPORTED
    assert "TC_BF16" in N.lib.frg_last_error().decode()
    assert code(lambda: frg.Matcher(unit, metric="euclidean").range_host(q, 0.5, -1, 4, variant="tc_exact")) == N.ERR_UNSUPPORTED
    bf = frg.GalleryStore(dim=d, capacity=64, bf16_only=True)
    bf.append_rows(np.eye(8, d, dtype=np.float32))
    assert code(lambda: frg.Matcher(bf).range_host(q, 0.5, -1, 4)) == N.ERR_UNSUPPORTED
    empty = frg.GalleryStore(dim=d, capacity=64)
    for v in ("auto", "tc_exact", "scan_f32"):
        c, r, s = frg.Matcher(empty).range_host(q, 0.5, -1, 3, variant=v)
        assert (c == 0).all() and (r == -1).all() and (s == -1.0).all()
    c, r, s = m.range_host(np.zeros((0, d), np.float32), 0.5, -1, 3)
    assert c.shape == (0,)
    # Euclidean: the exact scan, against the reference
    rng = np.random.default_rng(5)
    n = 30_000
    G = (rng.standard_normal((n, d)) * 0.1).astype(np.float32)
    raw = frg.GalleryStore(dim=d, capacity=n, raw=True)
    raw.append_rows(G)
    Q = np.concatenate([G[:3] + 0.01, (rng.standard_normal((20, d)) * 0.1).astype(np.float32)])
    for v in ("auto", "scan_f32"):
        c, r, s, name = raw_range(frg, raw, Q, 1.38, 4000, v, metric="euclidean")       # ~2 % of the rows
        assert name == "range_scan" and c.max() <= 4000 and c.sum() > 100 * len(Q)
        check_against_reference(c, r, s, Q, G, 1.38, metric="euclidean")
        assert (s[r < 0] == np.inf).all()
    for st in (unit, bf, empty, raw):
        st.close()


def test_python_layers(frg):
    from facerecognition_infrenceengine_b200.sharded import ShardedGallery, ShardedMatcher
    n, d = 200_000, 512
    store = frg.GalleryStore(dim=d, capacity=n)
    store.fill_synthetic(n, 0, synth.GALLERY_SEED)
    G = synth.gallery(n, d)
    Q, _ = synth.queries(64, n, d)
    m = frg.Matcher(store)
    res = m.match_range(Q, 0.16, max_hits=2)
    assert res.variant == "range_tc" and (res.counts > 2).any()
    ref_c, ref_r, ref_s = range_search(Q, G, 0.16)
    S = mo.cosine_scores(Q, G)
    for f in range(len(Q)):
        near = set(np.nonzero(np.abs(S[f] - np.float32(0.16)) <= NEAR)[0].tolist())
        assert set(res.rows[f].tolist()) - near == set(ref_r[f].tolist()) - near
        assert len(res.rows[f]) == res.counts[f] and res.ids[f] == store.ids_of(res.rows[f][None])[0]
        key = list(zip(-res.scores[f], res.rows[f]))
        assert key == sorted(key)                                                  # best first
    g = ShardedGallery(dim=d, store=store, rank=0, world=1)
    g.plan(n)
    sh = ShardedMatcher(g).match_range(Q, 0.16, max_hits=2, with_ids=False)
    assert np.array_equal(sh.counts, res.counts)
    for f in range(len(Q)):
        assert np.array_equal(sh.rows[f], res.rows[f]) and np.array_equal(sh.scores[f], res.scores[f])
    store.close()


def _planted(n, d, n_pairs, seed):
    rng = np.random.default_rng(seed)
    G = synth.gallery(n, d, seed)
    pairs = []
    src = rng.choice(n, 2 * n_pairs, replace=False)
    for a, b in zip(src[:n_pairs], src[n_pairs:]):
        G[b] = mo.normalise(G[a] + 0.3 * synth.gallery(1, d, int(b) + 100)[0])
        pairs.append((min(a, b), max(a, b)))
    return G, pairs


def _reference_pairs(G, ids, thr, mask):
    Gn = mo.normalise_rows(G)
    out = {}
    rows = np.nonzero(mask)[0]
    for a0 in range(0, len(rows), 2000):
        qa = rows[a0:a0 + 2000]
        S = mo.cosine_scores(G[qa], Gn)
        for i, a in enumerate(qa):
            hit = np.nonzero((S[i] > np.float32(thr)) & mask & (np.arange(len(G)) > a))[0]
            for b in hit:
                if ids[a] != ids[b]:
                    out[(ids[a], ids[b])] = float(S[i, b])
    return out


def test_duplicate_audit(frg):
    n, d = 20_000, 512
    G, planted = _planted(n, d, 50, 41)
    ids = ["id%05d" % i for i in range(n)]
    comp = ["acme" if (i // 1000) % 2 else "globex" for i in range(n)]
    store = frg.GalleryStore(dim=d, capacity=n)
    store.upsert(ids, G, comp)
    for company in (None, "acme"):
        mask = np.ones(n, bool) if company is None else np.array([c == company for c in comp])
        want = _reference_pairs(G, ids, 0.4, mask)
        got = frg.find_duplicate_pairs(store, 0.4, company_id=company, batch=1024)
        assert {(a, b) for a, b, _ in got} == set(want) and len(got) == len(want)
        for a, b, s in got:
            assert abs(s - want[(a, b)]) <= 1e-6
        if company is None:
            assert len(want) >= 50 and {(ids[a], ids[b]) for a, b in planted} <= set(want)
    store.close()
    # enrolment gallery: several templates of one person are not duplicates of each other
    eg = frg.EnrolmentGallery(dim=d, capacity=64)
    E = synth.gallery(6, d, 77)
    E[1] = E[0]
    E[4] = E[3]
    eg.add(["doc%d" % i for i in range(6)], E, ["acme"] * 6, ["employee"] * 6,
           ref_ids=["emp0", "emp0", "emp2", "emp3", "emp4", "emp5"])
    ck = frg.EnrolmentChecker(eg)
    got = ck.audit_duplicates("acme", "employee")
    assert [(a, b) for a, b, _ in got] == [("emp3", "emp4")]
    assert ck.audit_duplicates("acme", "visitor") == []
    eg.close()
