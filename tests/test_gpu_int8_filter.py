"""The int8 tensor-core filter of unit cosine stores: rows that saturate the store's int8 scale, the integer floor at
threshold edges, and no query handed to the exact fallback at the benchmark's shape (1 M x 512, 1024 queries)."""
import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frg():
    import facerecognition_infrenceengine_b200 as m
    return m


def same(a, b):
    assert np.array_equal(a.rows, b.rows)
    assert np.array_equal(a.scores.view(np.uint32), b.scores.view(np.uint32))
    assert np.array_equal(a.accept, b.accept)


def test_saturated_rows_match_the_exact_scan(frg):
    """Rows with elements far above the store scale (0.165 at dim 512) are clamped to +-127; their residual widens
    the bound, so the results still equal the exact scan's bit for bit - including for queries aimed at them."""
    n, d = 20000, 512
    store = frg.GalleryStore(dim=d, capacity=n + 8)
    store.fill_synthetic(n, 0, synth.GALLERY_SEED)
    rng = np.random.default_rng(7)
    spikes = np.zeros((4, d), np.float32)
    spikes[0, 3] = 1.0                                    # one element at 1.0: 6x the scale
    spikes[1, :4] = 0.5                                   # four at 0.5
    spikes[2] = rng.standard_normal(d).astype(np.float32)
    spikes[2, 10] = 40.0                                  # one dominant element among ordinary ones
    spikes[3, ::2] = 1.0                                  # flat: 0.0625 per element, no saturation
    store.append_rows(spikes)
    Q, _ = synth.queries(64, n, d)
    Qs = np.concatenate([Q, spikes + 0.05 * rng.standard_normal((4, d)).astype(np.float32)])
    m = frg.Matcher(store)
    for k in (1, 5):
        tc = m.match(Qs, k, 0.3, variant="tc_exact")
        assert tc.variant == "tc_exact"
        ex = m.match(Qs, k, 0.3, variant="scan_f32")
        same(tc, ex)
        assert (tc.rows[64:, 0] == np.arange(n, n + 4)).all()
    store.close()


def test_integer_floor_at_threshold_edges(frg):
    """Range search with the threshold set exactly to a row's exact score: that row is in (>=) or out (strict),
    identically on the int8 filter and on the exact counting scan."""
    n, d = 50000, 512
    store = frg.GalleryStore(dim=d, capacity=n)
    store.fill_synthetic(n, 0, synth.GALLERY_SEED)
    Q, _ = synth.queries(32, n, d)
    m = frg.Matcher(store)
    top = m.match(Q, 16, 0.3, variant="scan_f32")
    for j in (0, 4, 15):
        for f in range(0, 32, 8):
            thr = float(top.scores[f, j])
            for strict in (False, True):
                tc = m.range_host(Q[f:f + 1], thr, -1, 32, strict, "tc_exact")
                assert frg._native.last_variant() == "range_tc"
                ex = m.range_host(Q[f:f + 1], thr, -1, 32, strict, "scan_f32")
                for a, b in zip(tc, ex):
                    assert np.array_equal(a, b), (j, f, strict)
                hit = int(top.rows[f, j]) in set(tc[1][0, :tc[0][0]].tolist())
                assert hit != strict, (j, f, strict)
    store.close()


def test_no_fallback_at_the_benchmark_shape(frg):
    """1 M x 512 synthetic gallery, the benchmark's 1024 queries, top-5: every query is settled by the int8 filter
    and the select stage.  A query handed to the exact fallback would read the whole 2 GB master (>= 0.26 ms on a
    B200); with none the fallback stage is one idle launch."""
    n, d = 1_000_000, 512
    store = frg.GalleryStore(dim=d, capacity=n)
    store.fill_synthetic(n, 0, synth.GALLERY_SEED)
    Q, target = synth.queries(1024, n, d)
    m = frg.Matcher(store)
    ex = m.match(Q, 5, frg.CAMPUS_THRESHOLD, variant="scan_f32")
    for F in (1024, 256, 128, 64, 1):
        m.match(Q[:F], 5, frg.CAMPUS_THRESHOLD)           # warm-up
        frg._native.profile_enable(True)
        r = m.match(Q[:F], 5, frg.CAMPUS_THRESHOLD)
        frg._native.profile_collect()
        stages = frg._native.profile_stages()
        frg._native.profile_enable(False)
        assert r.variant == "tc_exact"
        assert stages["fallback"] < 0.1, (F, stages)
        assert np.array_equal(r.rows, ex.rows[:F]), F
        assert np.array_equal(r.scores.view(np.uint32), ex.scores[:F].view(np.uint32)), F
    store.close()
