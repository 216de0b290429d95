"""The int8 pre-pass packs each row group's winning 32-row block into 8 bits of its key, so a CTA that visits more
than one window of blocks (32 tiles in the CTA-pair form) publishes every window's maxima on its own.  At 3 M rows and
1024 queries each pre-pass CTA pair visits ~41 sampled tiles, ~9 of them in its second window.

What catches a wrong window -> row mapping is the fallback stage: the floor kernel rescores the row a key names, so a
key whose row lies in the wrong tile brings in an ordinary row of its group (exact score ~0 +- 0.05 instead of ~0.2).
e_k drops to about that score, the floor admits most of the gallery, and the query's candidate list overflows into the
exact fallback.  With ~22 % of the sampled tiles in second windows, most of the 1024 queries have at least one of their
5 best group winners there.  The results must equal the exact scan's bit for bit, with no query handed to the
fallback."""
import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu


def test_prepass_over_several_windows_matches_the_exact_scan():
    import facerecognition_infrenceengine_b200 as frg
    import torch
    n, d = 3_000_000, 512
    # tc_plan at 1024 queries: 4 pair columns, chunks_pre = (SMs / 2) / 4, sampled tiles = every 16th of the 256-row tiles
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    tiles_pre = -(-(-(-n // 256)) // 16)
    assert tiles_pre // ((sms // 2) // 4) > 32, "the pre-pass CTAs would not reach a second window"
    store = frg.GalleryStore(dim=d, capacity=n)
    store.fill_synthetic(n, 0, synth.GALLERY_SEED)
    Q, target = synth.queries(1024, n, d)
    m = frg.Matcher(store)
    ex = m.match(Q, 5, frg.CAMPUS_THRESHOLD, variant="scan_f32")
    m.match(Q, 5, frg.CAMPUS_THRESHOLD)                   # warm-up
    frg._native.profile_enable(True)
    r = m.match(Q, 5, frg.CAMPUS_THRESHOLD)
    frg._native.profile_collect()
    stages = frg._native.profile_stages()
    frg._native.profile_enable(False)
    assert r.variant == "tc_exact"
    assert stages["fallback"] < 0.1, stages
    assert np.array_equal(r.rows, ex.rows)
    assert np.array_equal(r.scores.view(np.uint32), ex.scores.view(np.uint32))
    assert np.array_equal(r.accept, ex.accept)
    assert (r.rows[target >= 0, 0] == target[target >= 0]).all()
    store.close()
