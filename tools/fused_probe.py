"""Top-k step time of a bf16-only store at small batches, device-timed without stage events (run on the GPU box).
Up to 8 queries run the fused probe+filter kernel, larger batches the separate pre-pass and filter.
    python tools/fused_probe.py [k] [batches...]"""
import sys

import torch

sys.path.insert(0, ".")
import facerecognition_infrenceengine_b200 as frg
from oracle import synth

n, d = 1_000_000, 512
k = int(sys.argv[1]) if len(sys.argv) > 1 else 5
batches = [int(a) for a in sys.argv[2:]] or [1, 8, 16, 32, 64, 128]
store = frg.GalleryStore(dim=d, capacity=n, bf16_only=True)
store.fill_synthetic(n, 0, 1234)
m = frg.Matcher(store)
for F in batches:
    Q = torch.from_numpy(synth.queries(F, n, d)[0]).cuda()
    out = None
    for _ in range(10):
        out = m.match_device(Q, k, 0.45, out=out)
    torch.cuda.synchronize()
    ts = []
    for rep in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            m.match_device(Q, k, 0.45, out=out)
        e1.record()
        torch.cuda.synchronize()
        ts.append(round(e0.elapsed_time(e1) / 50 * 1e3, 1))
    print("F=%4d k=%d step us %s" % (F, k, ts), flush=True)
