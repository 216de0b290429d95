"""Range search against top-k, and the whole-gallery duplicate audit, on one GPU (1 M x 512 synthetic gallery).

    python tools/range_probe.py --out profiles/r03_range_probe.json

Part 1: frg_match_range (threshold 0.4, max_hits 16) and frg_match top-5 (threshold 0.4) on the same device queries
at F = 1, 64 and 1024, timed with CUDA events over windows of back-to-back calls, the two alternating window by window
after a sustained warm-up (the card at its power-limited clocks, as bench.py measures).  Part 2: find_duplicate_pairs
over the gallery with planted near-duplicate pairs: wall time (profiling off) and device time (the library's per-stage
events, a second run), and 2 * N^2 * D flop over the device time.  The card's name, power limit and SM clocks are
read in the same run and written next to the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

BF16_DENSE_TFLOPS = 2250.0      # NVIDIA HGX B200 data sheet, one GPU, dense, at up to 1000 W


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--pairs", type=int, default=1000)
    a = ap.parse_args()
    import torch
    import facerecognition_infrenceengine_b200 as frg
    from facerecognition_infrenceengine_b200 import _native as N
    from oracle import matcher_oracle as mo
    from oracle import synth

    assert torch.cuda.is_available(), "no CUDA device: nothing to measure"
    n, d = a.rows, 512
    res = {"card_before": card(), "rows": n, "dim": d}
    store = frg.GalleryStore(dim=d, capacity=n)
    store.fill_synthetic(n, 0, synth.GALLERY_SEED)
    m = frg.Matcher(store)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    Qh, _ = synth.queries(1024, n, d)
    Qd = torch.from_numpy(Qh).to(dev)

    def topk_call(Q, out):
        m.match_device(Q, 5, 0.4, out=out)

    def range_call(Q, out):
        p = frg.matcher._params("cosine", "auto", 0.4, -1, 0)
        c, r, s = out
        N.check(N.lib.frg_match_range(store.handle, C.c_void_p(Q.data_ptr()), Q.shape[0], 16, C.byref(p),
                                      C.c_void_p(c.data_ptr()), C.c_void_p(r.data_ptr()), C.c_void_p(s.data_ptr()),
                                      C.c_void_p(stream.cuda_stream)))

    # sustained regime: a few seconds of the heaviest shape first
    F = 1024
    o_t = (torch.empty((F, 5), dtype=torch.int64, device=dev), torch.empty((F, 5), device=dev),
           torch.empty(F, dtype=torch.uint8, device=dev))
    t0 = time.time()
    while time.time() - t0 < 5.0:
        topk_call(Qd, o_t)
    torch.cuda.synchronize()
    part1 = {}
    for F, iters in ((1, 400), (64, 200), (1024, 40)):
        Q = Qd[:F].contiguous()
        o_t = (torch.empty((F, 5), dtype=torch.int64, device=dev), torch.empty((F, 5), device=dev),
               torch.empty(F, dtype=torch.uint8, device=dev))
        o_r = (torch.empty(F, dtype=torch.int64, device=dev), torch.empty((F, 16), dtype=torch.int64, device=dev),
               torch.empty((F, 16), device=dev))
        runs = {"topk5": (topk_call, o_t), "range_max16": (range_call, o_r)}
        for fn, o in runs.values():
            for _ in range(5):
                fn(Q, o)
        times = {k: [] for k in runs}
        for _ in range(a.rounds):
            for name, (fn, o) in runs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(iters):
                    fn(Q, o)
                e1.record(stream)
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) / iters)
        range_call(Q, o_r)
        torch.cuda.synchronize()
        part1["F=%d" % F] = {
            name: {"median_ms": float(np.median(t)), "min_ms": float(min(t)), "max_ms": float(max(t)), "windows": t}
            for name, t in times.items()}
        part1["F=%d" % F]["range_variant"] = N.last_variant()
        part1["F=%d" % F]["range_over_topk"] = part1["F=%d" % F]["range_max16"]["median_ms"] / part1["F=%d" % F]["topk5"]["median_ms"]
        part1["F=%d" % F]["mean_count"] = float(o_r[0].float().mean().item())
        print("F=%4d  top-5 %.4f ms  range %.4f ms  (x%.3f)" % (F, part1["F=%d" % F]["topk5"]["median_ms"],
              part1["F=%d" % F]["range_max16"]["median_ms"], part1["F=%d" % F]["range_over_topk"]), flush=True)
    res["range_vs_topk"] = part1

    # planted near-duplicate pairs: row b := normalise(row a + 0.3 * noise), cos ~ 0.96
    rng = np.random.default_rng(5)
    src = rng.choice(n, 2 * a.pairs, replace=False)
    pa, pb = src[:a.pairs], src[a.pairs:]
    A = np.stack([store.read_rows(int(r), 1)[0][0] for r in pa])
    B = mo.normalise_rows(A + 0.3 * mo.normalise_rows(rng.standard_normal(A.shape).astype(np.float32)))
    store.overwrite_rows(pb, B)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pairs = frg.find_duplicate_pairs(store, 0.4, batch=1024, matcher=m)
    wall = time.perf_counter() - t0
    found = {(int(x, 16), int(y, 16)) for x, y, _ in pairs}
    want = {(int(min(x, y)), int(max(x, y))) for x, y in zip(pa, pb)}
    N.lib.frg_profile_enable(1)
    frg.find_duplicate_pairs(store, 0.4, batch=1024, matcher=m)
    N.profile_collect()
    stages = N.profile_stages()
    N.lib.frg_profile_enable(0)
    dev_s = sum(stages.values()) / 1e3
    flop = 2.0 * n * n * d
    res["audit"] = {
        "rows": n, "planted": a.pairs, "pairs_found": len(pairs), "planted_found": len(want & found),
        "wall_s": wall, "device_s": dev_s, "device_stage_ms": stages,
        "flop": flop, "tflops_over_device_time": flop / dev_s / 1e12,
        "share_of_datasheet_bf16_dense": flop / dev_s / 1e12 / BF16_DENSE_TFLOPS,
        "note": "device time = summed per-stage CUDA events of the range calls (query prep, filter, select, "
                "fallback); wall time includes reading the rows back and the host-side pair assembly"}
    print("audit: %d rows, %d pairs (%d/%d planted), wall %.2f s, device %.3f s, %.0f TFLOP/s" % (
        n, len(pairs), len(want & found), a.pairs, wall, dev_s, flop / dev_s / 1e12), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    store.close()


if __name__ == "__main__":
    main()
