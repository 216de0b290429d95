"""Mixed-company range search on one B200: one frg_match_range per tenant (a) against one frg_match_range_tenants (b),
with one unfiltered frg_match_range of the same queries (c) for scale, and the batched enrolment duplicate check
(run on the GPU box):
    python tools/range_tenants_probe.py --out profiles/r09_range_tenants_probe.json

Gallery: 1 M x 512 synthetic rows, 100 contiguous companies of 10 000 rows (int8 plane).  Workloads: T tenants x f faces
(T in 1, 8, 64; f in 1, 4, 16), threshold 0.4, max_hits 16; and the exact path (SCAN_F32) at T = 64 x f = 4.  The arms
alternate in one process after a warm-up of every shape; each sample is device-event time over `--calls` calls.  (a)
and (b) are checked to be bit-identical in the same run.  The working set (0.5 GB int8 plane + 2 GB master) exceeds L2.
Enrolment check: 256 faces over 64 companies against a 100 k-row EnrolmentGallery (200 companies x 2 kinds of 250 rows),
plane-less and with an int8 plane: one check_duplicate_faces against 256 check_duplicate_face calls, host wall time of
whole calls (each ends in a device synchronise), results checked equal.
"""
import argparse
import ctypes as C
import json
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import facerecognition_infrenceengine_b200 as frg  # noqa: E402
from facerecognition_infrenceengine_b200 import _native as N  # noqa: E402
from facerecognition_infrenceengine_b200.enrol import EnrolmentChecker, EnrolmentGallery  # noqa: E402
from oracle import synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="profiles/r09_range_tenants_probe.json")
ap.add_argument("--calls", type=int, default=20)
ap.add_argument("--samples", type=int, default=7)
args = ap.parse_args()

n, d, T, H, THR = 1_000_000, 512, 10_000, 16, 0.4
store = frg.GalleryStore(dim=d, capacity=n)
for t0 in range(0, n, T):
    store.fill_synthetic(T, t0, synth.GALLERY_SEED, tag=1 + t0 // T)
torch.cuda.synchronize()
stream = torch.cuda.current_stream().cuda_stream


def params(tenant, variant):
    return N.MatchParams(N.METRIC_COSINE, N.VARIANTS[variant], float(np.float32(THR)), int(tenant), 0, 0, 0)


def ptr(t):
    return C.c_void_p(t.data_ptr())


def outputs(F):
    return [torch.empty(F, dtype=torch.int64, device="cuda"), torch.empty((F, H), dtype=torch.int64, device="cuda"),
            torch.empty((F, H), dtype=torch.float32, device="cuda")]


def workload(n_t, f, seed, variant="auto"):
    rng = np.random.default_rng(seed)
    ten = rng.choice(np.arange(1, n // T + 1), n_t, replace=False)
    tenants = np.repeat(ten, f).astype(np.int32)
    rows = (tenants - 1) * T + rng.integers(0, T, len(tenants))
    Q = synth.unit_rows(rows, d) + np.float32(0.03) * rng.standard_normal((len(rows), d)).astype(np.float32)
    order = rng.permutation(len(Q))
    Q, tenants = np.ascontiguousarray(Q[order], np.float32), tenants[order]
    groups = {}
    for i, t in enumerate(tenants.tolist()):
        groups.setdefault(t, []).append(i)
    Qd = torch.from_numpy(Q).cuda()
    sub = {t: (torch.from_numpy(np.ascontiguousarray(Q[ix])).cuda(), ix) for t, ix in groups.items()}
    F = len(Q)
    out = outputs(F)
    outs_a = {t: outputs(len(ix)) for t, (_, ix) in sub.items()}
    pa = {t: params(t, variant) for t in sub}
    pb = params(-1, variant)

    def arm_a():
        for t, (q, ix) in sub.items():
            o = outs_a[t]
            N.check(N.lib.frg_match_range(store.handle, ptr(q), len(ix), H, C.byref(pa[t]), ptr(o[0]), ptr(o[1]),
                                          ptr(o[2]), C.c_void_p(stream)))

    def arm_b():
        N.check(N.lib.frg_match_range_tenants(store.handle, ptr(Qd), F, H, C.byref(pb), tenants.ctypes.data,
                                              ptr(out[0]), ptr(out[1]), ptr(out[2]), C.c_void_p(stream)))

    def arm_c():
        N.check(N.lib.frg_match_range(store.handle, ptr(Qd), F, H, C.byref(pb), ptr(out[0]), ptr(out[1]),
                                      ptr(out[2]), C.c_void_p(stream)))

    def check():
        arm_a()
        arm_b()
        torch.cuda.synchronize()
        ok = True
        for t, (_, ix) in sub.items():
            ix = torch.tensor(ix, device="cuda")
            ok &= bool(torch.equal(out[0][ix], outs_a[t][0])) and bool(torch.equal(out[1][ix], outs_a[t][1]))
            ok &= bool(torch.equal(out[2][ix].view(torch.int32), outs_a[t][2].view(torch.int32)))
        return ok
    return dict(F=F, tenants=len(sub), a=arm_a, b=arm_b, c=arm_c, check=check)


def timed(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls * 1e3          # us per call


shapes = []
for n_t in (1, 8, 64):
    for f in (1, 4, 16):
        shapes.append(("T%d_f%d" % (n_t, f), workload(n_t, f, 100 * n_t + f)))
shapes.append(("scan_f32_T64_f4", workload(64, 4, 11, variant="scan_f32")))

for _, w in shapes:                                     # warm-up of every shape and arm
    for arm in "abc":
        w[arm]()
torch.cuda.synchronize()

results = {}
all_same = True
for name, w in shapes:
    same = w["check"]()
    all_same &= same
    samples = {"a": [], "b": [], "c": []}
    for _ in range(args.samples):
        for arm in "abc":
            samples[arm].append(timed(w[arm], args.calls))
    w["b"]()
    launches, variant = N.last_launch_count(), N.last_variant()
    res = {"F": w["F"], "tenants": w["tenants"], "bit_identical_a_b": same, "b_variant": variant, "b_launches": launches}
    for arm in "abc":
        v = sorted(samples[arm])
        res[arm + "_us"] = {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}
    res["b_over_a"] = res["b_us"]["median"] / res["a_us"]["median"]
    results[name] = res
    print("%-18s F=%4d a=%8.1f b=%7.1f c=%7.1f us  b/a=%.3f  same=%s %s launches=%d" % (
        name, w["F"], res["a_us"]["median"], res["b_us"]["median"], res["c_us"]["median"], res["b_over_a"], same,
        variant, launches), flush=True)
store.close()

# ---- the batched enrolment duplicate check
enrol = {}
ne, per_company = 100_000, 250
rng = np.random.default_rng(3)
G = rng.standard_normal((ne, d)).astype(np.float32)
companies = ["co%d" % (i // (2 * per_company)) for i in range(ne)]
kinds = ["employee" if (i // per_company) % 2 == 0 else "visitor" for i in range(ne)]
pick = rng.choice(ne, 256, replace=False)
cos = sorted(set(companies[p] for p in pick))[:64]
pick = np.array([p for p in rng.permutation(ne) if companies[p] in cos][:256])
E = G[pick] + np.float32(0.3) * rng.standard_normal((len(pick), d)).astype(np.float32)
E[::2] = rng.standard_normal((len(E[::2]), d)).astype(np.float32)             # half of them new people
cids, ks = [companies[p] for p in pick], [kinds[p] for p in pick]
for plane in (False, True):
    eg = EnrolmentGallery(store=frg.GalleryStore(dim=d, capacity=ne, bf16_plane=plane))
    eg.add(["doc%d" % i for i in range(ne)], G, companies, kinds)
    chk = EnrolmentChecker(eg)
    batched = lambda: chk.check_duplicate_faces(E, cids, ks)                                   # noqa: E731
    single = lambda: [chk.check_duplicate_face(E[i], cids[i], ks[i]) for i in range(len(E))]  # noqa: E731
    same = batched() == single()
    all_same &= same
    tb, ts = [], []
    for _ in range(args.samples):
        t0 = time.perf_counter()
        batched()
        tb.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        single()
        ts.append((time.perf_counter() - t0) * 1e3)
    tb.sort()
    ts.sort()
    dups = int(sum(r[0] for r in batched()))
    name = "enrolment_%s" % ("int8_plane" if plane else "no_plane")
    enrol[name] = {"faces": len(E), "companies": len(set(cids)), "duplicates": dups,
                   "same_results": same, "batched_variant": N.last_variant(),
                   "batched_ms": {"median": tb[len(tb) // 2], "min": tb[0], "max": tb[-1]},
                   "per_face_ms": {"median": ts[len(ts) // 2], "min": ts[0], "max": ts[-1]}}
    print("%-22s batched %.2f ms (%s)  per-face loop %.2f ms  same=%s" % (
        name, tb[len(tb) // 2], enrol[name]["batched_variant"], ts[len(ts) // 2], same), flush=True)
    eg.close()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
doc = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": smi,
       "gallery": "1M x 512 synthetic, 100 contiguous companies of 10000 rows", "threshold": THR, "max_hits": H,
       "calls_per_sample": args.calls, "samples": args.samples,
       "arms": {"a": "one frg_match_range per tenant, one stream", "b": "one frg_match_range_tenants",
                "c": "one unfiltered frg_match_range of the same queries"},
       "results": results, "enrolment_check": enrol}
with open(args.out, "w") as fh:
    json.dump(doc, fh, indent=1)
print(smi)
assert all_same, "the arms disagree"
