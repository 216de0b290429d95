"""BASELINE config 1 on the GPU (run on the GPU box): 10 000 x 512 gallery, frames of F faces, top-1 + threshold,
one frg_match_host call per frame (host buffers in and out, result waited for) and device-timed.
    python tools/config1_probe.py [rows] [variant]"""
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import facerecognition_infrenceengine_b200 as frg
from oracle import matcher_oracle as mo
from oracle import synth

n = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000
variant = sys.argv[2] if len(sys.argv) > 2 else "auto"
d = 512
store = frg.GalleryStore(dim=d, capacity=n)
store.fill_synthetic(n, 0, synth.GALLERY_SEED)
G, _ = store.read_rows()
m = frg.Matcher(store)
for F in (1, 8, 64, 256):
    Q, _ = synth.queries(F, n, d)
    ref = mo.match_topk(Q, G, 2, 0.45)
    for _ in range(30):
        r = m.match(Q, 1, 0.45, variant=variant, with_ids=False)
    assert mo.ids_match_with_gap(ref[0], ref[1], r.rows, 1e-4).all() and (r.accept == ref[2]).all()
    t0 = time.perf_counter()
    for _ in range(300):
        r = m.match(Q, 1, 0.45, variant=variant, with_ids=False)
    e2e_us = (time.perf_counter() - t0) / 300 * 1e6
    Qd = torch.from_numpy(Q).cuda()
    out = None
    for _ in range(30):
        out = m.match_device(Qd, 1, 0.45, variant=variant, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(300):
        m.match_device(Qd, 1, 0.45, variant=variant, out=out)
    e1.record()
    torch.cuda.synchronize()
    print("rows=%d F=%4d variant=%s(%s) launches=%d  e2e %.1f us/frame  device %.1f us/frame" % (
        n, F, variant, r.variant, r.launches, e2e_us, e0.elapsed_time(e1) / 300 * 1e3), flush=True)
store.close()
