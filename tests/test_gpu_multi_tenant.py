"""frg_match_tenants: one call in which every query carries its own tenant filter.  Every result is compared bit for
bit (rows, scores, accept) with frg_match of that query alone with its own tenant - the existing, oracle-pinned path."""
import ctypes as C

import numpy as np
import pytest

from oracle import matcher_oracle as mo
from oracle import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frg():
    import facerecognition_infrenceengine_b200 as m
    return m


def _params(N, tenant=-1, variant="auto", threshold=0.4, metric="cosine"):
    return N.MatchParams(N.METRICS[metric], N.VARIANTS[variant], float(np.float32(threshold)), int(tenant), 0, 0, 0)


def tenants_call(store, Q, tenants, k, **kw):
    from facerecognition_infrenceengine_b200 import _native as N
    Q = np.ascontiguousarray(Q, np.float32)
    F = len(Q)
    t = np.ascontiguousarray(tenants, np.int32)
    rows, scores, acc = np.empty((F, k), np.int64), np.empty((F, k), np.float32), np.zeros(F, np.uint8)
    p = _params(N, **kw)
    N.check(N.lib.frg_match_tenants_host(store.handle, Q.ctypes.data, F, k, C.byref(p), t.ctypes.data,
                                         rows.ctypes.data, scores.ctypes.data, acc.ctypes.data))
    return rows, scores, acc, N.last_variant(), N.last_launch_count()


def per_query(store, Q, tenants, k, **kw):
    """frg_match of every query alone, with its own tenant"""
    from facerecognition_infrenceengine_b200 import _native as N
    F = len(Q)
    rows, scores, acc = np.empty((F, k), np.int64), np.empty((F, k), np.float32), np.zeros(F, np.uint8)
    for i in range(F):
        q = np.ascontiguousarray(Q[i:i + 1], np.float32)
        p = _params(N, tenant=int(tenants[i]), **kw)
        N.check(N.lib.frg_match_host(store.handle, q.ctypes.data, 1, k, C.byref(p), rows[i:].ctypes.data,
                                     scores[i:].ctypes.data, acc[i:].ctypes.data))
    return rows, scores, acc


def check(store, Q, tenants, k, variant_ran=None, **kw):
    r, s, a, var, launches = tenants_call(store, Q, tenants, k, **kw)
    rr, rs, ra = per_query(store, Q, tenants, k, **kw)
    assert np.array_equal(r, rr)
    assert np.array_equal(s.view(np.uint32), rs.view(np.uint32))
    assert np.array_equal(a, ra)
    if variant_ran is not None:
        assert var == variant_ran
    return r, s, a, launches


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


@pytest.mark.parametrize("k", [1, 5, 16])
def test_many_tenants_one_call(big, k):
    Q, tenants = company_queries(64, 15, 1, extra_all=40, extra_unknown=24)
    assert len(Q) == 1024
    r, s, a, _ = check(big, Q, tenants, k, variant_ran="tc_exact_grouped")
    assert (r[tenants == 777] == -1).all() and not a[tenants == 777].any()
    # ids of one tenant against the oracle on that tenant's rows only
    t = int(tenants[0])
    sel = tenants == t
    G, _ = big.read_rows((t - 1) * T, T)
    ref = mo.match_topk(Q[sel], G, k + 1, 0.4)
    want = np.where(ref[0] >= 0, ref[0] + (t - 1) * T, -1)
    assert mo.ids_match_with_gap(want, ref[1], r[sel], 1e-4).all()


def test_launch_count_does_not_grow_with_tenants(big):
    counts = []
    for n_t in (8, 64):
        Q, tenants = company_queries(n_t, 4, n_t)
        *_, launches = check(big, Q, tenants, 5, variant_ran="tc_exact_grouped")
        counts.append(launches)
    assert counts[0] == counts[1]


def test_single_tenant_is_frg_match(big, frg):
    from facerecognition_infrenceengine_b200 import _native as N
    Q, _ = company_queries(1, 40, 3)
    tenants = np.full(len(Q), 5, np.int32)
    r, s, a, var, _ = tenants_call(big, Q, tenants, 5)
    m = frg.Matcher(big).match(Q, 5, 0.4, company_id="c5")
    assert var == m.variant
    assert np.array_equal(r, m.rows) and np.array_equal(s.view(np.uint32), m.scores.view(np.uint32))
    assert np.array_equal(a.view(bool), m.accept)
    # all "all tenants" queries: the unfiltered frg_match
    check(big, Q[:3], [-1, -5, -1], 3)


def test_stretched_company_and_overflow(frg):
    """a company re-enrolled once at the gallery's end (tile list), and a company whose rows are hundreds of
    near-duplicates of its queries (candidate overflow -> exact fallback with the query's own tenant)"""
    n = 300_000
    store = frg.GalleryStore(dim=DIM, capacity=n + 1024)
    for t0 in range(0, n, T):
        store.fill_synthetic(T, t0, synth.GALLERY_SEED, tag=1 + t0 // T)
    rng = np.random.default_rng(5)
    store.overwrite_rows([n - 1], synth.unit_rows([n - 1], DIM), np.array([7], np.int32), prenormalised=True)
    base = synth.unit_rows([3 * T + 17], DIM)[0]
    dups = base[None, :] + np.float32(1e-3) * rng.standard_normal((600, DIM)).astype(np.float32)
    store.append_rows(dups, np.full(600, 4, np.int32))           # tenant 4: its block + 600 near-duplicates
    Qs, ts = [], []
    for t in (7, 4, 9, 12, -1):
        rows = (abs(t) - 1) * T + rng.integers(0, T, 6) if t > 0 else rng.integers(0, n, 6)
        Qs.append(synth.unit_rows(rows, DIM) + np.float32(0.02) * rng.standard_normal((6, DIM)).astype(np.float32))
        ts += [t] * 6
    Qs.append(np.repeat(base[None, :], 4, 0) + np.float32(1e-3) * rng.standard_normal((4, DIM)).astype(np.float32))
    ts += [4] * 4
    Q = np.concatenate(Qs).astype(np.float32)
    perm = rng.permutation(len(Q))
    for k in (1, 16):
        check(store, Q[perm], np.array(ts, np.int32)[perm], k, variant_ran="tc_exact_grouped")
    store.close()


def test_layouts(frg):
    """tiny companies, interleaved companies (scattered tags: masked range), tombstones, NaN rows and queries,
    compaction between two calls, nq = 0 and 1"""
    rng = np.random.default_rng(11)
    n = 40_000
    store = frg.GalleryStore(dim=256, capacity=n + 4096)
    G = rng.standard_normal((n, 256)).astype(np.float32)
    tags = np.where(np.arange(n) < 20_000, np.arange(n) % 3 + 1, 10 + (np.arange(n) - 20_000) // 100).astype(np.int32)
    store.append_rows(G, tags)                                    # 1..3 interleaved, then 200 companies of 100 rows
    nanrow = np.full((1, 256), np.nan, np.float32)
    store.append_rows(nanrow, np.array([12], np.int32))
    store.remove_rows(rng.integers(0, n, 500))
    tq = np.array([1, 2, 3, 10, 11, 150, 209, -1, 999, 12] * 6, np.int32)
    rows = np.array([np.nonzero(tags == t)[0][i % 50] if t in tags else 0 for i, t in enumerate(tq)])
    Q = G[rows] + np.float32(0.1) * rng.standard_normal((len(tq), 256)).astype(np.float32)
    Q[5] = np.nan
    for k in (1, 4):
        check(store, Q, tq, k, variant_ran="tc_exact_grouped")
    check(store, Q[:0], tq[:0], 3)
    check(store, Q[:1], tq[:1], 3)
    store.compact()
    check(store, Q, tq, 5, variant_ran="tc_exact_grouped")
    store.close()


def test_device_written_tags_and_empty_gallery(frg):
    """tags upserted from device arrays (the store's tenant extents become unknown: every tile, masked); an empty
    gallery gives every query row -1 / reject"""
    import torch
    from facerecognition_infrenceengine_b200 import _native as N
    store = frg.GalleryStore(dim=128, capacity=8192)
    Q = np.random.default_rng(2).standard_normal((20, 128)).astype(np.float32)
    t = np.array([1, 2, -1, 3] * 5, np.int32)
    r, s, a, *_ = check(store, Q, t, 3)
    assert (r == -1).all() and not a.any()
    rng = np.random.default_rng(3)
    G = torch.from_numpy(rng.standard_normal((6000, 128)).astype(np.float32)).cuda()
    tags = torch.from_numpy((np.arange(6000) // 2000 + 1).astype(np.int32)).cuda()
    N.check(N.lib.frg_store_upsert(store.handle, None, C.c_void_p(G.data_ptr()), C.c_void_p(tags.data_ptr()), 6000,
                                   0, None))
    torch.cuda.synchronize()
    Q = G[::300].cpu().numpy() + np.float32(0.05)
    check(store, Q, (np.arange(len(Q)) % 4).astype(np.int32) - 1 + 1, 5, variant_ran="tc_exact_grouped")
    store.close()


# ------------------------------------------------------------------ stores and variants served by the per-tenant loop
def test_loop_path_stores(frg):
    rng = np.random.default_rng(9)
    n = 20_000
    G = rng.standard_normal((n, 128)).astype(np.float32)
    tags = (np.arange(n) // 5000 + 1).astype(np.int32)
    Q = G[rng.integers(0, n, 24)] + np.float32(0.05) * rng.standard_normal((24, 128)).astype(np.float32)
    tq = np.array([1, 2, 3, 4, -1, 8] * 4, np.int32)
    stores = {
        "plain": frg.GalleryStore(dim=128, capacity=n),
        "raw": frg.GalleryStore(dim=128, capacity=n, raw=True),
        "bf16_only": frg.GalleryStore(dim=128, capacity=n, bf16_only=True),
        "no_plane": frg.GalleryStore(dim=128, capacity=n, bf16_plane=False),
    }
    for s in stores.values():
        s.append_rows(G, tags)
    check(stores["plain"], Q, tq, 5, variant="scan_f32", variant_ran="scan_f32")
    check(stores["raw"], G[:24] * 3 + 0.1, tq, 5, metric="euclidean", threshold=0.6)
    check(stores["bf16_only"], Q, tq, 5)
    check(stores["no_plane"], Q, tq, 5, variant_ran="scan_f32")
    for s in stores.values():
        s.close()


# ------------------------------------------------------------------ Python
def test_python_layers(frg):
    import torch
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
    cids = [comp[p] if i % 4 else ("globex" if i % 8 == 0 else None) for i, p in enumerate(pick)]
    cids[3] = "nobody"
    r = m.match_tenants(Q, cids, k=3)
    assert r.variant == "tc_exact_grouped"
    for i in range(len(Q)):
        one = m.match(Q[i:i + 1], 3, company_id=cids[i])
        assert np.array_equal(one.rows[0], r.rows[i]) and one.ids[0] == r.ids[i] and one.accept[0] == r.accept[i]
    assert r.ids[3] == [None, None, None]
    # device tensors on a non-default stream
    st = torch.cuda.Stream()
    Qd = torch.from_numpy(Q).cuda()
    codes = [-1 if c is None else store.tenant_code(c, create=False) for c in cids]
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        rows, scores, acc = m.match_tenants_device(Qd, codes, k=3, stream=st.cuda_stream)
    st.synchronize()
    assert np.array_equal(rows.cpu().numpy(), r.rows) and np.array_equal(acc.cpu().numpy().view(bool), r.accept)
    # recognize_frames == recognize frame by frame
    proc = frg.FaceRecognitionProcessor(store)
    frames = [(Q[0:5], "acme"), (Q[5:5], "globex"), (Q[5:12], None), (Q[12:20], "initech"), (Q[20:22], "nobody")]
    got = proc.recognize_frames(frames)
    want = [proc.recognize(e, c) for e, c in frames]
    assert [[(x["person_id"], float(x["recognition_score"])) for x in f] for f in got] == \
           [[(x["person_id"], float(x["recognition_score"])) for x in f] for f in want]
    # the aggregator mixes companies in one batch through match_many_fn
    from facerecognition_infrenceengine_b200.aggregator import BatchAggregator

    def many(Qb, companies):
        res = m.match_tenants(Qb, companies, k=1, with_ids=False)
        return res.rows, res.scores, res.accept

    agg = BatchAggregator(None, max_batch=64, max_delay_ms=50, match_many_fn=many)
    futs = [agg.submit(e, c) for e, c in frames if len(e)]
    res = [f.result(timeout=30) for f in futs]
    agg.close()
    for (e, c), (rows_, scores_, acc_) in zip([fr for fr in frames if len(fr[0])], res):
        one = m.match(e, 1, company_id=c)
        assert np.array_equal(rows_, one.rows) and np.array_equal(acc_, one.accept)
    store.close()
