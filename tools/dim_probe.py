"""Per-stage device timings of the cosine TC pipeline for other row lengths (run on the GPU box).
    python tools/dim_probe.py rows dim k batch [batch ...]
"""
import json
import sys

import torch

sys.path.insert(0, ".")
import facerecognition_infrenceengine_b200 as frg
from facerecognition_infrenceengine_b200 import _native as N
from oracle import synth

n, d, k = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
store = frg.GalleryStore(dim=d, capacity=n)
store.fill_synthetic(n, 0, 1234)
m = frg.Matcher(store)
for F in [int(a) for a in sys.argv[4:]]:
    Q = torch.from_numpy(synth.queries(F, n, d)[0]).cuda()
    out = None
    for _ in range(5):
        out = m.match_device(Q, k, 0.45, out=out)
    torch.cuda.synchronize()
    N.profile_enable(True)
    N.profile_collect()
    steps = 30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        m.match_device(Q, k, 0.45, out=out)
    e1.record()
    torch.cuda.synchronize()
    N.profile_collect()
    st = {a: round(b / steps * 1e3, 1) for a, b in N.profile_stages().items()}
    N.profile_enable(False)
    dom = st["dominant"] * 1e-6
    print(json.dumps({"rows": n, "dim": d, "k": k, "batch": F, "step_us_with_events": round(e0.elapsed_time(e1) / steps * 1e3, 1),
                      "stages_us": st, "filter_GBs": round(n * d * 2 / dom / 1e9, 1),
                      "filter_TFs": round(2.0 * F * n * d / dom / 1e12, 1)}), flush=True)
