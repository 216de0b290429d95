"""Per-stage device times of the int8 tensor-core filter (B200): prep, pre-pass, floor, filter, select and the exact
fallback, at batch sizes 1 / 64 / 128 / 256 / 1024 over the 1 M x 512 synthetic gallery, top-5.  A query the filter
hands to the exact fallback re-reads the whole 2 GB master (>= 0.26 ms on a B200), so a fallback stage at its idle
cost (a few microseconds) means no query was flagged; the stage times are read after the timed calls.

    python tools/int8_probe.py [--rows 1000000] [--reps 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import facerecognition_infrenceengine_b200 as frg  # noqa: E402
from facerecognition_infrenceengine_b200 import _native as N  # noqa: E402
from oracle import synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--batches", default="1,64,128,256,1024")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    store = frg.GalleryStore(dim=a.dim, capacity=a.rows)
    store.fill_synthetic(a.rows, 0, synth.GALLERY_SEED)
    Q, _ = synth.queries(1024, a.rows, a.dim)
    m = frg.Matcher(store)
    res = {"gpu": gpu, "rows": a.rows, "dim": a.dim, "k": 5, "batches": {}}
    for F in [int(x) for x in a.batches.split(",")]:
        q = np.ascontiguousarray(Q[:F])
        for _ in range(3):
            m.match(q, 5, frg.CAMPUS_THRESHOLD, with_ids=False)
        t0 = time.perf_counter()
        for _ in range(a.reps):
            r = m.match(q, 5, frg.CAMPUS_THRESHOLD, with_ids=False)
        wall = (time.perf_counter() - t0) / a.reps * 1e3
        N.profile_enable(True)
        N.profile_collect()
        for _ in range(a.reps):
            m.match(q, 5, frg.CAMPUS_THRESHOLD, with_ids=False)
        N.profile_collect()
        st = {k_: v / a.reps for k_, v in N.profile_stages().items()}
        N.profile_enable(False)
        res["batches"][str(F)] = {"variant": r.variant, "call_ms": wall, "stage_ms": st,
                                  "fallback_idle": st["fallback"] < 0.1}
        print(F, json.dumps(res["batches"][str(F)]), flush=True)
    store.close()
    txt = json.dumps(res, indent=1)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
