#!/usr/bin/env python
"""Time UnknownClusterer.observe_batch (one frg_cluster_observe_host per batch) against the per-face loop it
replaces (one frg_first_match_host + host mean + upsert per face), whole calls with host wall time after a warm-up.
    python tools/cluster_probe.py --out profiles/r10_cluster_probe.json [--reps 5]

Grid: C0 existing clusters x B faces per batch, for two face mixes:
  join: half the faces are new views of existing clusters (score ~0.8, they join), half are new people;
  new:  every face is a new person (founds a cluster) - the resolve kernel's worst case (a dot per touched cluster).
Both arms start from the same clusters and observe the same batches; their results must be identical.  The stage
split (pre-pass = the range scan, resolve = the one-CTA kernel) comes from a separate, profiled call."""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import deque

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import facerecognition_infrenceengine_b200 as frg  # noqa: E402
from facerecognition_infrenceengine_b200 import _native as N  # noqa: E402
from cluster_streams import PerFaceClusterer  # noqa: E402

DIM = 512


def unit_rows(a):
    return (a / np.linalg.norm(a, axis=1, keepdims=True)).astype(np.float32)


def batch_of(rng, C0, B, mix):
    new = unit_rows(rng.standard_normal((B, DIM)))
    if mix == "new" or len(C0) == 0:
        return new
    old = unit_rows(C0[rng.integers(0, len(C0), B)] + 0.03 * rng.standard_normal((B, DIM)))
    return np.where((np.arange(B) % 2 == 0)[:, None], old, new).astype(np.float32)


def same_state(uc, ref):
    a, b = uc.representatives(), ref.store.read_rows()[0]
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)) and \
        uc.detection_count == ref.detection_count


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r10_cluster_probe.json")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    rng = np.random.default_rng(1)
    results, all_same = [], True
    for c0 in (100, 1000, 10000):
        C0 = unit_rows(rng.standard_normal((c0, DIM)))
        for mix in ("join", "new"):
            uc, ref = frg.UnknownClusterer(dim=DIM), PerFaceClusterer(dim=DIM)
            uc.observe_batch(C0)                                   # random directions: c0 clusters of one face
            ref.store.append_rows(C0, np.zeros(c0, np.int32))
            for q in C0:
                ref.members.append(deque([q], maxlen=10))
                ref.detection_count.append(1)
            for warm in batch_of(rng, C0, 4, mix):                 # modules, pinned buffers, allocator pools
                uc.observe_batch(warm[None])
                ref.observe(warm)
            same = same_state(uc, ref)
            for B in (1, 16, 256, 1024):
                tb, tl = [], []
                for _ in range(args.reps):
                    Q = batch_of(rng, C0, B, mix)
                    t0 = time.perf_counter()
                    got = uc.observe_batch(Q)
                    t1 = time.perf_counter()
                    want = [ref.observe(q) for q in Q]
                    t2 = time.perf_counter()
                    tb.append((t1 - t0) * 1e3)
                    tl.append((t2 - t1) * 1e3)
                    same &= got == want
                # stage split of one more batch: device time of the pre-pass and of the resolve kernel
                Q = batch_of(rng, C0, B, mix)
                N.profile_enable(True)
                got = uc.observe_batch(Q)
                N.profile_collect()
                stages = N.profile_stages()
                N.profile_enable(False)
                same &= got == [ref.observe(q) for q in Q]
                same &= same_state(uc, ref)
                all_same &= same
                tb.sort()
                tl.sort()
                row = {"c0": c0, "mix": mix, "B": B, "clusters_at_end": len(uc), "same_results": bool(same),
                       "batched_ms": {"median": tb[len(tb) // 2], "min": tb[0], "max": tb[-1]},
                       "per_face_ms": {"median": tl[len(tl) // 2], "min": tl[0], "max": tl[-1]},
                       "prepass_device_ms": stages["prepass"], "resolve_device_ms": stages["dominant"]}
                results.append(row)
                print("C0=%5d %-4s B=%4d  batched %8.3f ms  per-face %8.3f ms  (pre-pass %.3f, resolve %.3f ms) same=%s"
                      % (c0, mix, B, row["batched_ms"]["median"], row["per_face_ms"]["median"],
                         stages["prepass"], stages["dominant"], same), flush=True)
            uc.close()
            ref.close()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    doc = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": smi,
           "dim": DIM, "threshold": 0.65, "window": 10, "reps": args.reps,
           "arms": {"batched": "UnknownClusterer.observe_batch: one frg_cluster_observe_host",
                    "per_face": "frg_first_match_host + host np.mean + frg_store_upsert_host per face"},
           "timing": "host wall time of whole calls (each ends in a device synchronise), median of reps",
           "results": results}
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(smi)
    assert all_same, "the arms disagree"


if __name__ == "__main__":
    main()
