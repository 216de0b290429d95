"""Mixed-company batches on one B200: one frg_match per tenant (a) against one frg_match_tenants (b), with one
unfiltered frg_match of the same queries (c) for scale (run on the GPU box):
    python tools/multi_tenant_probe.py --out profiles/r06_multi_tenant_probe.json

Gallery: 1 M x 512 synthetic rows, 100 contiguous companies of 10 000 rows.  Workloads: T tenants x f faces (T in 1, 8,
64; f in 1, 4, 16), k = 5, threshold 0.4; a mixed batch (512 unfiltered queries + 64 companies x 4 faces); a stretched
company (one row re-enrolled at the gallery's end, as tools/tenant_probe.py far).  The arms alternate in one process
after a warm-up of every shape; each sample is device-event time over `--calls` calls.  (a) and (b) are checked to be
bit-identical in the same run.  The working set (0.5 GB int8 plane + 2 GB master) exceeds L2.
"""
import argparse
import ctypes as C
import json
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import facerecognition_infrenceengine_b200 as frg  # noqa: E402
from facerecognition_infrenceengine_b200 import _native as N  # noqa: E402
from oracle import synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="profiles/r06_multi_tenant_probe.json")
ap.add_argument("--calls", type=int, default=20)
ap.add_argument("--samples", type=int, default=7)
args = ap.parse_args()

n, d, T, k = 1_000_000, 512, 10_000, 5
store = frg.GalleryStore(dim=d, capacity=n)
for t0 in range(0, n, T):
    store.fill_synthetic(T, t0, synth.GALLERY_SEED, tag=1 + t0 // T)
torch.cuda.synchronize()
stream = torch.cuda.current_stream().cuda_stream


def params(tenant):
    return N.MatchParams(N.METRIC_COSINE, N.VARIANT_AUTO, float(np.float32(0.4)), int(tenant), 0, 0, 0)


def workload(n_t, f, seed, extra_all=0, stretched=False):
    rng = np.random.default_rng(seed)
    ten = rng.choice(np.arange(1, n // T + 1), n_t, replace=False)
    if stretched:
        ten[0] = 37
    tenants = np.repeat(ten, f).astype(np.int32)
    rows = (tenants - 1) * T + rng.integers(0, T, len(tenants))
    Q = synth.unit_rows(rows, d) + np.float32(0.03) * rng.standard_normal((len(rows), d)).astype(np.float32)
    if extra_all:
        Qa, _ = synth.queries(extra_all, n, d)
        Q = np.concatenate([Q, Qa])
        tenants = np.concatenate([tenants, np.full(extra_all, -1, np.int32)])
    order = rng.permutation(len(Q))
    Q, tenants = np.ascontiguousarray(Q[order], np.float32), tenants[order]
    groups = {}
    for i, t in enumerate(tenants.tolist()):
        groups.setdefault(t, []).append(i)
    Qd = torch.from_numpy(Q).cuda()
    sub = {t: (torch.from_numpy(np.ascontiguousarray(Q[ix])).cuda(), ix) for t, ix in groups.items()}
    F = len(Q)
    out = [torch.empty((F, k), dtype=torch.int64, device="cuda"), torch.empty((F, k), dtype=torch.float32, device="cuda"),
           torch.empty(F, dtype=torch.uint8, device="cuda")]
    outs_a = {t: [torch.empty((len(ix), k), dtype=torch.int64, device="cuda"),
                  torch.empty((len(ix), k), dtype=torch.float32, device="cuda"),
                  torch.empty(len(ix), dtype=torch.uint8, device="cuda")] for t, (_, ix) in sub.items()}
    pa = {t: params(t) for t in sub}
    pb, pc = params(-1), params(-1)

    def arm_a():
        for t, (q, ix) in sub.items():
            o = outs_a[t]
            N.check(N.lib.frg_match(store.handle, C.c_void_p(q.data_ptr()), len(ix), k, C.byref(pa[t]),
                                    C.c_void_p(o[0].data_ptr()), C.c_void_p(o[1].data_ptr()),
                                    C.c_void_p(o[2].data_ptr()), C.c_void_p(stream)))

    def arm_b():
        N.check(N.lib.frg_match_tenants(store.handle, C.c_void_p(Qd.data_ptr()), F, k, C.byref(pb),
                                        tenants.ctypes.data, C.c_void_p(out[0].data_ptr()),
                                        C.c_void_p(out[1].data_ptr()), C.c_void_p(out[2].data_ptr()),
                                        C.c_void_p(stream)))

    def arm_c():
        N.check(N.lib.frg_match(store.handle, C.c_void_p(Qd.data_ptr()), F, k, C.byref(pc),
                                C.c_void_p(out[0].data_ptr()), C.c_void_p(out[1].data_ptr()),
                                C.c_void_p(out[2].data_ptr()), C.c_void_p(stream)))

    def check():
        arm_a()
        arm_b()
        torch.cuda.synchronize()
        ok = True
        for t, (_, ix) in sub.items():
            ix = torch.tensor(ix, device="cuda")
            ok &= bool(torch.equal(out[0][ix], outs_a[t][0])) and bool(torch.equal(out[2][ix], outs_a[t][2]))
            ok &= bool(torch.equal(out[1][ix].view(torch.int32), outs_a[t][1].view(torch.int32)))
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
shapes.append(("mixed_512all_T64_f4", workload(64, 4, 7, extra_all=512)))
store.overwrite_rows([n - 1], synth.unit_rows([n - 1], d), np.array([37], np.int32), prenormalised=True)
shapes.append(("stretched_T8_f4", workload(8, 4, 9, stretched=True)))

for _, w in shapes:                                     # warm-up of every shape and arm
    for arm in "abc":
        w[arm]()
torch.cuda.synchronize()

results = {}
for name, w in shapes:
    same = w["check"]()
    samples = {"a": [], "b": [], "c": []}
    for _ in range(args.samples):
        for arm in "abc":
            samples[arm].append(timed(w[arm], args.calls))
    # per-stage split of (b), a run of its own
    N.profile_enable(True)
    for _ in range(args.calls):
        w["b"]()
    N.profile_collect()
    stages = {s: v * 1e3 / args.calls for s, v in N.profile_stages().items()}
    N.profile_enable(False)
    w["b"]()
    launches, variant = N.last_launch_count(), N.last_variant()
    res = {"F": w["F"], "tenants": w["tenants"], "bit_identical_a_b": same, "b_variant": variant, "b_launches": launches,
           "b_stage_us": stages}
    for arm in "abc":
        v = sorted(samples[arm])
        res[arm + "_us"] = {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}
    res["b_over_a"] = res["b_us"]["median"] / res["a_us"]["median"]
    results[name] = res
    print("%-22s F=%4d a=%8.1f b=%7.1f c=%7.1f us  b/a=%.3f  same=%s %s launches=%d" % (
        name, w["F"], res["a_us"]["median"], res["b_us"]["median"], res["c_us"]["median"], res["b_over_a"], same,
        variant, launches), flush=True)

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
doc = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": smi,
       "gallery": "1M x 512 synthetic, 100 contiguous companies of 10000 rows", "k": k, "threshold": 0.4,
       "calls_per_sample": args.calls, "samples": args.samples,
       "arms": {"a": "one frg_match per tenant, one stream", "b": "one frg_match_tenants",
                "c": "one unfiltered frg_match of the same queries"},
       "results": results}
with open(args.out, "w") as fh:
    json.dump(doc, fh, indent=1)
print(smi)
store.close()
