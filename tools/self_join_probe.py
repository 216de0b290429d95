#!/usr/bin/env python
"""Duplicate audit: the device self-join (find_duplicate_pairs / audit_duplicates / within_companies) against the
readback path (rows copied to the host and sent back as range-search queries), in one run, on the same stores.
    python tools/self_join_probe.py [--out profiles/r07_self_join_probe.json] [--rows 1000000]
Workloads: a 1 M x 512 store with an int8 scan plane and 1000 planted pairs (cos ~ 0.96, as tools/range_probe.py),
strict threshold 0.4; the same size in 100 contiguous companies of 10 000 rows (one within_companies pass against
100 audit_duplicates calls; the readback path only for the first 3 companies - it copies the whole gallery per
company); a 100 k-row plane-less enrolment gallery.  Both arms must return identical pair lists."""
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
from facerecognition_infrenceengine_b200.enrol import _find_duplicate_pairs_readback  # noqa: E402
from oracle import matcher_oracle as mo  # noqa: E402
from oracle import synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True).stdout.strip()
    return q


def planted(n, d, n_pairs, seed, plane=True, companies=1):
    store = frg.GalleryStore(dim=d, capacity=n, bf16_plane=plane)
    block = n // companies
    for t in range(companies):
        store.fill_synthetic(block, t * block, synth.GALLERY_SEED, tag=t)
        store._tenants["c%d" % t] = t
    rng = np.random.default_rng(seed)
    A = rng.choice(n, n_pairs, replace=False)
    B = []
    for a in A.tolist():             # the copy sits in its source's company
        lo = (a // block) * block
        b = a
        while b == a or b in B or b in A:
            b = int(rng.integers(lo, lo + block))
        B.append(b)
    vecs = []
    for a, b in zip(A.tolist(), B):
        v, _ = store.read_rows(a, 1)
        vecs.append(mo.normalise(v[0] + 0.3 * synth.gallery(1, d, b + 100)[0]))
    _, tb = store.read_rows(0, n)
    store.overwrite_rows(B, np.stack(vecs), tb[B])
    return store


def timed(fn, profile):
    import torch
    torch.cuda.synchronize()
    if profile:
        N.lib.frg_profile_enable(1)
        N.profile_collect()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t
    stages = None
    if profile:
        ms, launches = N.profile_collect()
        stages = dict(N.profile_stages(), launches=launches)
        N.lib.frg_profile_enable(0)
    return out, wall, stages


def arms(name, new_fn, old_fn, res):
    new, t_new, _ = timed(new_fn, False)
    old, t_old, _ = timed(old_fn, False)
    _, _, s_new = timed(new_fn, True)
    _, _, s_old = timed(old_fn, True)
    same = new == old
    res[name] = {"self_join_wall_s": t_new, "readback_wall_s": t_old, "speedup": t_old / t_new,
                 "self_join_stage_ms": s_new, "readback_stage_ms": s_old, "pairs": len(new) if isinstance(new, list) else None,
                 "identical": bool(same)}
    print(name, json.dumps(res[name]), flush=True)
    assert same, name


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07_self_join_probe.json")
    ap.add_argument("--rows", type=int, default=1_000_000)
    args = ap.parse_args()
    n, d = args.rows, 512
    res = {"card_before": card(), "rows": n, "dim": d, "threshold": 0.4, "strict": True}
    # warm every kernel shape once
    w = planted(20_000, d, 50, 1)
    frg.find_duplicate_pairs(w, 0.4)
    _find_duplicate_pairs_readback(w, 0.4)
    w.close()

    store = planted(n, d, 1000, 7)
    arms("whole_gallery_1M_int8_plane", lambda: frg.find_duplicate_pairs(store, 0.4),
         lambda: _find_duplicate_pairs_readback(store, 0.4), res)
    store.close()

    store = planted(n, d, 1000, 8, companies=100)
    ck = frg.EnrolmentChecker(store)
    one, t_one, s_one = timed(lambda: frg.find_duplicate_pairs(store, 0.4, within_companies=True), False)
    loop, t_loop, _ = timed(lambda: [frg.find_duplicate_pairs(store, 0.4, company_id="c%d" % t) for t in range(100)],
                            False)
    every, t_every, _ = timed(ck.audit_all_duplicates, False)
    _, _, s_one = timed(lambda: frg.find_duplicate_pairs(store, 0.4, within_companies=True), True)
    rb, t_rb, _ = timed(lambda: [_find_duplicate_pairs_readback(store, 0.4, "c%d" % t) for t in range(3)], False)
    assert sorted(one) == sorted(p for ps in loop for p in ps)
    assert all(every["c%d" % t] == loop[t] for t in range(100))
    assert all(rb[t] == loop[t] for t in range(3))
    res["companies_100x10k"] = {
        "within_companies_pass_s": t_one, "audit_all_duplicates_s": t_every, "loop_100_audit_duplicates_s": t_loop,
        "readback_3_companies_s": t_rb, "readback_per_company_s": t_rb / 3,
        "readback_100_companies_extrapolated_s": t_rb / 3 * 100, "within_stage_ms": s_one, "pairs": len(one),
        "identical": True}
    print("companies", json.dumps(res["companies_100x10k"]), flush=True)
    store.close()

    eg = frg.EnrolmentGallery(dim=d, capacity=100_000, store=planted(100_000, d, 200, 9, plane=False))
    arms("enrolment_100k_no_plane", lambda: frg.find_duplicate_pairs(eg, 0.4),
         lambda: _find_duplicate_pairs_readback(eg, 0.4), res)
    eg.close()
    res["card_after"] = card()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
