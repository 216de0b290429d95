#!/usr/bin/env python
"""Benchmark of the embedding-vs-gallery matching path (BASELINE.json metric: face queries/s at a
1 M x 512 gallery, top-5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch F]
                    [--dump-outputs DIR] ...

One "step" = one batch of F query embeddings matched against the whole resident gallery
(normalise -> scan -> top-k -> threshold).  Prints ONE JSON line (see DESIGN.md "Measurement").
  value     device-timed (CUDA events) whole-job queries/s, inputs already in HBM
  e2e       the same through the host-buffer C-ABI call (frg_match_host): pinned host queries in,
            H2D + kernels + D2H of ids/scores/decisions inside the timed region
  roofline  dominant kernel: algorithmic bytes (or flops) / its CUDA-event time vs the measured peak
  cpu_baseline  the reference's per-face Python loop (oracle port) on the host cores, bounded sample
--impl reference times only that CPU loop, on all host cores.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "face queries/sec at 1Mx512 gallery top-5"
UNIT = "queries/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        # drop the first sample (taken while the GPU was still ramping up)
        under = sm[1:] if len(sm) > 2 else sm
        return {"sm_mhz": float(np.median(under)) if under else None, "sm_max_mhz": max(mx) if mx else None,
                "sm_mhz_min": min(under) if under else None, "samples": len(sm), "reasons": sorted(reasons),
                "window": "identical load for ~1 s immediately before + the timed region"}


# ------------------------------------------------------------------------------------ CPU baseline
_G = None


def _cpu_worker(args):
    """The reference's per-face loop (oracle port of infrenceServer.py:530-552 / peopleCount.py:860-887)."""
    q_block, threshold = args
    from oracle import matcher_oracle as mo
    ids, emb = _G
    t0 = time.perf_counter()
    out = []
    for e in q_block:
        q = mo.normalise(e)
        bid, bs = mo.scan_best(q, emb)
        out.append((bid, float(bs), bool(bid and bs >= threshold)))
    return out, time.perf_counter() - t0


def _gen_rows(args):
    a, b, dim, seed = args
    from oracle import synth
    return a, synth.gallery(b - a, dim, seed, row0=a)


def cpu_gallery(n, dim, seed, procs):
    """frg-synth-v1 gallery on the host (bit-identical to the device generator), generated in parallel."""
    from multiprocessing import shared_memory
    out = np.empty((n, dim), np.float32)
    step = max(1, (n + procs * 4 - 1) // (procs * 4))
    jobs = [(a, min(n, a + step), dim, seed) for a in range(0, n, step)]
    with mp.get_context("fork").Pool(procs) as pool:
        for a, rows in pool.imap_unordered(_gen_rows, jobs):
            out[a:a + len(rows)] = rows
    return out


def run_cpu_loop(G, Q, threshold, procs, steps, warmup):
    """Process-per-camera model of the reference (infrenceServer.py:640-646): `procs` workers, each
    matching its share of every batch with the verbatim per-face loop.  Returns (q/s, per-step s, results)."""
    global _G
    ids = ["%024x" % i for i in range(len(G))]
    _G = (ids, dict(zip(ids, G)))            # the reference's Dict[str, np.ndarray]; forked, not copied
    times, results = [], None
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        for it in range(warmup + steps):
            blocks = [b for b in np.array_split(Q, procs) if len(b)]
            t0 = time.perf_counter()
            res = pool.map(_cpu_worker, [(b, threshold) for b in blocks])
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
                results = [r for part, _ in res for r in part]
    _G = None
    per_step = float(np.mean(times))
    return len(Q) / per_step, per_step, results


# ------------------------------------------------------------------------------------ arms
def reference_arm(args, rank, world):
    """--impl reference: the reference's CPU matcher (oracle port; the reference itself is a Python
    script that cannot travel to the GPU box) on all host cores, on the same workload."""
    if rank != 0:
        return
    procs = args.cpu_procs or (os.cpu_count() or 1)
    n, dim = args.rows, args.dim
    t0 = time.perf_counter()
    G = cpu_gallery(n, dim, args.seed, procs)
    from oracle import synth
    # bounded sample: the per-face loop costs ~0.65 us per gallery row; 1..8 queries per worker per step so
    # that the whole --steps/--warmup run stays around 1.5 minutes
    per_query_s = max(n * 0.65e-6, 1e-4)
    per_worker = max(1, min(8, int(90.0 / ((args.steps + args.warmup) * per_query_s))))
    q_per_step = args.cpu_queries or procs * per_worker
    Q, _ = synth.queries(q_per_step, n, dim)
    gen_s = time.perf_counter() - t0
    qps, per_step, _ = run_cpu_loop(G, Q, 0.45, procs, args.steps, args.warmup)
    sample = "%d queries/step (%d worker processes) x %d rows, top-1 + threshold (the reference has no top-k)" % (
        q_per_step, procs, n)
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, args.batch, world),
            "cpu_baseline": {"value": qps, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample,
                             "sample_queries_per_step": q_per_step},
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "setup_s": gen_s}
    emit_json(line)


def workload_config(args, batch, world=1):
    cfg = {"workload": "configs[1]: 512-d cosine, 1M-template gallery, top-5, single B200",
           "gallery_rows": args.rows, "dim": args.dim, "batch": batch, "k": args.k, "threshold": 0.45,
           "variant": args.variant}
    if args.bf16_only:
        cfg["storage"] = "bf16-only gallery (FRG_STORE_BF16_ONLY): scores are the bf16 filter's, |dscore| <= eps[q] (~3.6e-3 for ordinary data, 7.9e-3 worst case)"
    if args.rows_total:
        cfg.update({"workload": "configs[3]: 512-d cosine, %d-template gallery row-sharded over %d B200 (%d rows each), "
                                "batch %d, top-%d, per-rank top-k exchanged and merged (config.exchange)" % (
                                    args.rows_total, world, args.rows, batch, args.k),
                    "sharding": "gallery rows", "gallery_rows_total": args.rows_total})
    elif world > 1 and args.shard == "gallery":
        cfg.update({"workload": "gallery_rows_total=%d: configs[1] per GPU (weak scaling) - one gallery of %d x %d rows "
                                "row-sharded over %d GPUs, every query of the batch matched against ALL of them, "
                                "per-rank top-k exchanged and merged" % (
                                    args.rows * world, world, args.rows, world),
                    "sharding": "gallery rows", "gallery_rows_total": args.rows * world,
                    "value_definition": "whole-job aggregate in the metric's own unit: `raw_queries_per_s` (batch / "
                                        "step time, against gallery_rows_total rows) x gallery_rows_total / 1M, i.e. a "
                                        "query matched against N x 1M rows counts as N queries at 1M x 512 - per-GPU "
                                        "work is fixed, so this is what grows with N under weak scaling"})
    elif world > 1:
        cfg.update({"workload": "configs[1] replicated on %d GPUs, query stream sharded across ranks, no collective" % world,
                    "sharding": "queries (replicas)"})
    cfg.update({
            "l2_policy": "inputs larger than L2 (gallery %.2f GB fp32 + %.2f GB bf16 plane vs 126 MB L2)" % (
                args.rows * args.dim * 4 / 1e9, args.rows * args.dim * 2 / 1e9)})
    return cfg


def power_capped(clocks):
    """The clock record of a timed region shows the power cap (or clocks well below max): the sustained cuBLAS
    figure is the tensor denominator for that region, the burst figure otherwise (B200_PROFILING.md)."""
    return bool(clocks and ("sw_power_cap" in (clocks.get("reasons") or []) or (
        clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and clocks["sm_mhz"] < 0.9 * clocks["sm_max_mhz"])))


def roofline_for(variant, n, dim, F, dom_launch_ms, peaks):
    """Roofline of the dominant kernel: t_roof = max(bytes / BW_hbm, flops / P_tensor) (SURVEY.md 8d).
    scan_f32 reads the fp32 master once per pass of <= 4 queries; the tcgen05 filter reads the bf16
    scan plane once per batch and does 2*F*n*dim flops."""
    if variant == "scan_f32":
        bytes_ = n * dim * 4
        ach = bytes_ / (dom_launch_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "scan_f32_kernel", "achieved": ach, "peak": peaks["hbm_gbs"],
                "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None,
                "algorithmic_bytes_per_launch": bytes_, "launch_ms": dom_launch_ms, "peak_source": peaks["source"]}
    return tc_roofline(variant, n, dim, F, dom_launch_ms, peaks)


def ours_arm(args, rank, world):
    import torch
    import facerecognition_infrenceengine_b200 as frg
    from facerecognition_infrenceengine_b200 import _native as N
    from oracle import matcher_oracle as mo
    from oracle import synth

    # the library's bound on a rank waiting for its peers is 2 s; a bench whose ranks also do unsynchronised host
    # work (allocating 150 GB, CPU spot checks) gives them 10 s before a skew is called a failure
    os.environ.setdefault("FRG_EXCHANGE_TIMEOUT_MS", "10000")
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    if args.rows_total:                      # BASELINE configs[3]: a FIXED gallery row-sharded over the ranks
        args.rows = args.rows_total // world
    n, dim, k = args.rows, args.dim, args.k

    sharded = world > 1 and args.shard == "gallery"
    # (slack: the config 5 leg enrols a few thousand rows at the end; growing would re-allocate the gallery)
    store = frg.GalleryStore(dim=dim, capacity=n + (16384 if world == 1 else 0), device=local, bf16_only=args.bf16_only)
    if sharded:
        from facerecognition_infrenceengine_b200.sharded import ShardedGallery, ShardedMatcher
        sg = ShardedGallery(dim=dim, device=local, store=store)
        sg.fill_synthetic(n * world, args.seed)          # this rank: rows [rank*n, (rank+1)*n)
        smatcher = ShardedMatcher(sg, exchange=args.exchange)
    else:
        store.fill_synthetic(n, 0, args.seed)
    torch.cuda.synchronize()
    matcher = frg.Matcher(store)
    stream = torch.cuda.current_stream(dev)
    nb = 4
    n_total = n * world if sharded else n
    # units of work per step: sharded -> every query is matched against world x n rows
    scale = 1.0 if args.rows_total else float(world)     # fixed gallery: plain queries/s (strong scaling)

    def make_batches(F):
        # a ring of distinct query batches (50 % genuine / 50 % impostor, SURVEY.md section 8d);
        # every rank takes its own slice of the query stream
        # (row-sharded: every rank needs the SAME batch; replicas: each rank its own slice)
        Qh = [synth.queries(F, n_total, dim, q0=((0 if sharded else rank) * nb + i) * F)[0] for i in range(nb)]
        Qd = [torch.from_numpy(q).to(dev) for q in Qh]
        outs = [(torch.empty((F, k), dtype=torch.int64, device=dev),
                 torch.empty((F, k), dtype=torch.float32, device=dev),
                 torch.empty((F,), dtype=torch.uint8, device=dev)) for _ in range(nb)]
        return Qh, Qd, outs

    def time_device(F, steps, warmup, Qd, outs, clocks=False, preload_s=None, keep_last=False):
        preload_s = args.clock_preload_s if preload_s is None else preload_s
        def step(i):
            if sharded:
                smatcher.match(Qd[i % nb], k, 0.45, variant=args.variant, out=outs[i % nb])
            else:
                matcher.match_device(Qd[i % nb], k, 0.45, variant=args.variant, out=outs[i % nb])
        for i in range(warmup):
            step(i)
        torch.cuda.synchronize()
        launches_per_step, variant = N.last_launch_count(), N.last_variant()
        sampler = None
        if clocks:
            # nvidia-smi samples every 100 ms: keep the GPU under the SAME load for ~1 s right before the
            # timed region (untimed), so that the clock / throttle record describes the state the timed
            # steps run in even when K steps last only milliseconds
            # step() is a COLLECTIVE on a row-sharded gallery: every rank must make the same number of calls.
            # (Round 1 looped on each rank's own wall clock: ranks left after different counts and the rank with
            # more calls polled for packets nobody would send.)  One block of 16 steps is timed, the slowest
            # rank's time fixes the block count for everybody.
            sampler = ClockSampler(local)
            sampler.start()
            t0 = time.perf_counter()
            for i in range(16):
                step(i)
            torch.cuda.synchronize()
            blk = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                torch.distributed.all_reduce(blk, op=torch.distributed.ReduceOp.MAX)
            nblk = int(min(4096, max(0, np.ceil(preload_s / max(float(blk.item()), 1e-6)) - 1)))
            for b in range(nblk):
                for i in range(16):
                    step(i)
                if b % 4 == 3:
                    torch.cuda.synchronize()
            torch.cuda.synchronize()
            if sharded:
                smatcher.check_exchange()
        # Inside the timed region only the DOMINANT kernel is bracketed by events, on every 4th step (an
        # event pair costs ~6 us of stream time; bracketing every stage ~30 us per step = 12 % at batch 64,
        # tools/event_tax_probe.py), so the per-stage split comes from a separate short pass below.
        N.check(N.lib.frg_profile_enable(3))
        N.profile_collect()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for i in range(steps):
            step(i)
        ev1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        total_ms = ev0.elapsed_time(ev1)
        dom_ms, dom_launches = N.profile_collect()
        ck = sampler.stop() if sampler else None
        # the passes below reuse the output buffers: copy the last timed step's results out first
        last = [x.cpu().numpy() for x in outs[(steps - 1) % nb]] if keep_last else None
        # per-stage split (untimed for `value`): every stage bracketed, a few steps
        N.check(N.lib.frg_profile_enable(1))
        nsplit = max(5, min(steps, 30))
        for i in range(nsplit):
            step(i)
        torch.cuda.synchronize()
        N.profile_collect()
        stages = {k_: v / nsplit for k_, v in N.profile_stages().items()}
        N.profile_enable(False)
        # spread of single steps (SURVEY.md section 8d: median, p10, p90): one event per step boundary
        nsp = max(10, min(steps, 100))
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(nsp + 1)]
        evs[0].record(stream)
        for i in range(nsp):
            step(i)
            evs[i + 1].record(stream)
        torch.cuda.synchronize()
        per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(nsp))
        spread = {"p10": per[nsp // 10], "p50": per[nsp // 2], "p90": per[(nsp * 9) // 10], "steps": nsp}
        if sharded:
            smatcher.check_exchange()                # a void collective call raises here, with the reason
        if world > 1:
            t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            total_ms = float(t.item())
        ms = total_ms / steps
        return {"batch": F, "value": F * scale / (ms * 1e-3), "ms_per_step": ms, "variant": variant,
                "launches_per_step": launches_per_step, "dom_ms": dom_ms, "dom_launches": dom_launches,
                "dom_steps": (steps + 3) // 4,          # steps whose dominant kernel was bracketed
                "total_ms": total_ms, "clocks": ck, "stage_ms": stages, "step_ms_spread": spread, "last": last}

    # ---- headline batch: device-timed region
    F = args.batch
    Qh, Qd, outs = make_batches(F)
    main = time_device(F, args.steps, args.warmup, Qd, outs, clocks=True, keep_last=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *main["last"])
    variant = main["variant"]
    clocks = main["clocks"]
    peaks["use_sustained"] = power_capped(clocks)
    ms_per_step, value = main["ms_per_step"], main["value"]

    # ---- the same batches with TWO in flight (two streams, alternating): what a server with two camera
    # threads gets on the device side - the small kernels of one batch (query prep, select, fallback) run
    # under the tensor-core filter of the other.  Reported beside `value`, never instead of it.
    pipelined = None
    if not sharded and world == 1 and args.steps >= 4:
        s2 = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
        for i in range(8):
            matcher.match_device(Qd[i % nb], k, 0.45, variant=args.variant, out=outs[i % nb],
                                 stream=s2[i % 2].cuda_stream)
        torch.cuda.synchronize()
        p0, p1a, p1b = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        p0.record(s2[0])
        s2[1].wait_event(p0)
        for i in range(args.steps):
            matcher.match_device(Qd[i % nb], k, 0.45, variant=args.variant, out=outs[i % nb],
                                 stream=s2[i % 2].cuda_stream)
        p1a.record(s2[0])
        p1b.record(s2[1])
        torch.cuda.synchronize()
        ms2 = max(p0.elapsed_time(p1a), p0.elapsed_time(p1b)) / args.steps
        pipelined = {"streams": 2, "value": F / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2, "steps": args.steps,
                     "note": "device-timed, two batches in flight on two streams; same kernels, same work per step"}

    # ---- parity spot-check of what was just timed (never inside the timed region).  Bounded: at most
    # CHECK_ROWS gallery rows are copied back to the host, whatever the gallery size.
    parity = None
    if not args.no_check and (sharded or rank == 0):
        CHECK_ROWS = 2_000_000
        m = min(n, CHECK_ROWS)
        nchk = min(F, 32 if m == n else 16)
        tol = 8e-3 if args.bf16_only else 1e-4
        Gs, _ = store.read_rows(0, m)                                   # this rank's first m rows
        off = sg.offset if sharded else 0
        sub_rows, sub_scores, sub_acc = mo.match_topk(Qh[0][:nchk], Gs, k + 1, 0.45)
        if sharded:
            torch.distributed.barrier()          # the host work above took a different time on every rank
            smatcher.match(Qd[0], k, 0.45, variant=args.variant, out=outs[0])
        else:
            matcher.match_device(Qd[0], k, 0.45, variant=args.variant, out=outs[0])
        torch.cuda.synchronize()
        if sharded:
            smatcher.check_exchange()
        got_r, got_s, got_a = (x.cpu().numpy() for x in outs[0])
        ok = True
        for f in range(nchk):
            # every checked row that clearly beats the returned k-th score must have been returned,
            # and the returned list is ordered
            must = sub_rows[f][(sub_rows[f] >= 0) & (sub_scores[f] >= got_s[f, k - 1] + tol)] + off
            ok &= set(must) <= set(got_r[f])
            ok &= bool(np.all(np.diff(got_s[f]) <= 0))
        parity = {"checked_queries": nchk, "checked_rows": m, "id_gap_tolerance": tol, "subset_ids_ok": bool(ok)}
        if m == n and not sharded:
            parity.update({"ids_ok": bool(mo.ids_match_with_gap(sub_rows, sub_scores, got_r[:nchk], tol).all()),
                           "max_abs_dscore": float(np.abs(got_s[:nchk] - sub_scores[:, :k]).max()),
                           "accept_ok": bool((got_a[:nchk].astype(bool) == sub_acc).all())})
        if sharded:
            t = torch.tensor([1.0 if ok else 0.0], device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MIN)
            parity["sharded_ids_ok_all_ranks"] = bool(t.item() > 0)
        del Gs

    # ---- end to end through the host-buffer ABI call (pinned host in, pinned host out)
    Qp = [torch.from_numpy(q).pin_memory() for q in Qh]
    rows_p = torch.empty((F, k), dtype=torch.int64).pin_memory()
    sc_p = torch.empty((F, k), dtype=torch.float32).pin_memory()
    ac_p = torch.empty((F,), dtype=torch.uint8).pin_memory()
    res = frg.MatchResult(rows_p.numpy(), sc_p.numpy(), ac_p.numpy())
    q_dev = torch.empty((F, dim), dtype=torch.float32, device=dev)

    def e2e_step(i):
        if sharded:
            # host batch in (pinned) -> H2D on every rank -> sharded match -> D2H of the merged result
            q_dev.copy_(Qp[i % nb], non_blocking=True)
            r_, s_, a_ = smatcher.match(q_dev, k, 0.45, variant=args.variant, out=outs[0])
            rows_p.copy_(r_, non_blocking=True); sc_p.copy_(s_, non_blocking=True); ac_p.copy_(a_, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        else:
            matcher.match(Qp[i % nb].numpy(), k, 0.45, variant=args.variant, with_ids=False, out=res)

    if world > 1:
        torch.distributed.barrier()
    for i in range(max(3, args.warmup)):
        e2e_step(i)
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item())
    if sharded:
        smatcher.check_exchange()
    e2e = {"value": F * scale * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": F * dim * 4,
           "d2h_bytes_per_step": F * k * 12 + F, "ms_per_step": e2e_s / args.steps * 1e3,
           "callers": 1,
           "api": ("ShardedMatcher.match: pinned host batch -> H2D -> frg_match per shard -> exchange + merge "
                   "(config.exchange) -> D2H" if sharded else
                   "frg_match_host via Matcher.match (pinned host buffers)")}

    # The reference runs one matcher thread per camera against one shared gallery (peopleCount.py:918-924):
    # the same public call from TWO host threads, each with its own batches and result buffers.  Every
    # step still copies its batch in and its results out inside the timed region; the copies and the
    # launch latency of one caller overlap the kernels of the other (frg_match_host is re-entrant: one
    # stream per host thread).  Reported beside the single-caller figure, never instead of it.
    if not sharded and args.e2e_callers > 1:
        import threading
        T = args.e2e_callers
        per = max(1, args.steps // T)
        start = threading.Barrier(T + 1)
        spans, errs = [None] * T, []

        def caller(ti):
            try:
                torch.cuda.set_device(local)
                Qt = [torch.from_numpy(q).pin_memory() for q in Qh]
                rt = frg.MatchResult(torch.empty((F, k), dtype=torch.int64).pin_memory().numpy(),
                                     torch.empty((F, k), dtype=torch.float32).pin_memory().numpy(),
                                     torch.empty((F,), dtype=torch.uint8).pin_memory().numpy())
                mt = frg.Matcher(store)
                for i in range(3):
                    mt.match(Qt[i % nb].numpy(), k, 0.45, variant=args.variant, with_ids=False, out=rt)
                start.wait()
                a = time.perf_counter()
                for i in range(per):
                    mt.match(Qt[(i + ti) % nb].numpy(), k, 0.45, variant=args.variant, with_ids=False, out=rt)
                spans[ti] = (a, time.perf_counter())
            except Exception as ex:          # noqa: BLE001
                errs.append(repr(ex))
                try:
                    start.abort()
                except Exception:            # noqa: BLE001
                    pass

        th = [threading.Thread(target=caller, args=(ti,)) for ti in range(T)]
        [t_.start() for t_ in th]
        try:
            start.wait()
        except threading.BrokenBarrierError:
            pass
        [t_.join() for t_ in th]
        if not errs and all(spans):
            wall = max(b for _, b in spans) - min(a for a, _ in spans)
            e2e["concurrent"] = {"callers": T, "value": F * per * T / wall, "unit": UNIT,
                                 "ms_per_step": wall / (per * T) * 1e3, "steps": per * T,
                                 "h2d_bytes_per_step": F * dim * 4, "d2h_bytes_per_step": F * k * 12 + F}
        else:
            e2e["concurrent"] = {"callers": T, "error": errs[:2]}

    # ---- other batch sizes of configs[1] ("batch 1-1024"): device-timed, same method
    sweep = []
    if args.sweep and world == 1 and not sharded:
        for Fs in [int(x) for x in args.sweep.split(",") if x]:
            if Fs == F:
                r = main
            else:
                _, Qd_s, outs_s = make_batches(Fs)
                # every point under its own ~0.5 s of identical load with its own clock record: a tensor-bound
                # batch settles on the power cap, an HBM-bound one does not - each fraction uses the peak of
                # the regime that point actually ran in
                r = time_device(Fs, args.steps, args.warmup, Qd_s, outs_s, clocks=True,
                                preload_s=min(args.clock_preload_s, 0.5))
                del Qd_s, outs_s
            pk = dict(peaks, use_sustained=power_capped(r["clocks"]))
            rf = roofline_for(r["variant"], n, dim, Fs, r["dom_ms"] / max(r["dom_launches"], 1), pk)
            ck = r["clocks"] or {}
            sweep.append({"batch": Fs, "value": r["value"], "ms_per_step": r["ms_per_step"], "variant": r["variant"],
                          "bound": rf["bound"], "kernel_frac": rf["frac"], "kernel_ms": rf["launch_ms"],
                          "peak": rf["peak"], "peak_kind": rf.get("peak_kind", "measured copy bandwidth"),
                          "sm_mhz": ck.get("sm_mhz"), "clock_reasons": ck.get("reasons"),
                          "stage_ms": {k_: round(v, 4) for k_, v in r["stage_ms"].items()},
                          "step_ms_spread": {k_: round(v, 4) for k_, v in r["step_ms_spread"].items()},
                          "step_frac_of_roofline": step_roofline_ms(n, dim, Fs, pk) / r["ms_per_step"]})

    # ---- BASELINE configs[3] ("config 4" in DESIGN.md's 1-based count): the FIXED 100 M x 512 gallery
    # row-sharded over the ranks, batch 4096, top-10, peer-memory exchange - every multi-GPU run carries it
    config4 = None
    if sharded and not args.rows_total and args.config4_rows > 0:
        config4 = run_config4(args, rank, world, local, dev, peaks)

    if rank != 0:
        return

    roof = roofline_for(variant, n, dim, F, main["dom_ms"] / max(main["dom_launches"], 1), peaks)
    roof["traffic"], roof["traffic_source"] = ncu_traffic(variant, n, dim, F, world)
    roof["launches_per_step"] = main["dom_launches"] / main["dom_steps"]
    roof["timed_launches"] = main["dom_launches"]
    roof["kernel_share_of_step"] = (main["dom_ms"] / main["dom_steps"]) / ms_per_step
    roof["step_frac_of_roofline"] = step_roofline_ms(n, dim, F, peaks) / ms_per_step

    # ---- CPU baseline (bounded sample of the same workload, on this box's host cores)
    cpu = None
    if not args.no_cpu:
        procs = args.cpu_procs or (os.cpu_count() or 1)
        if n > 4_000_000:
            raise SystemExit("cpu_baseline copies the gallery to the host: use --no-cpu above 4 M rows")
        G, _ = store.read_rows()                        # bit-identical to the CPU generator (tested)
        # ~10-15 s of wall clock on every core: 16 queries per worker at 1 M rows (~0.65 us per row and query)
        q_cpu = args.cpu_queries or procs * max(1, min(16, int(12.0 / max(n * 0.65e-6, 1e-4))))
        Qc, _ = synth.queries(q_cpu, n, dim)
        qps, per_step, results = run_cpu_loop(G, Qc, 0.45, procs, 1, 0)
        # the same queries through the GPU (rank 0's rows): identical ids and decisions
        r = matcher.match(Qc, 1, 0.45, variant=args.variant)
        same = all((res_[0] == gid[0] or (res_[0] is None and gid[0] is None)) and (res_[2] == bool(a))
                   for res_, gid, a in zip(results, r.ids, r.accept))
        # BASELINE config 1 as the reference runs it: 10 000 x 512 gallery, 64 faces, ONE core
        G1 = G[:10000]
        Q1, _ = synth.queries(64, 10000, dim)
        qps1, _, res1 = run_cpu_loop(G1, Q1, 0.45, 1, 1, 0)
        # ... and the same frame through the GPU, end to end from host buffers (frg_match_host), as the
        # reference's call site would use it: one call per frame, result waited for
        st1 = frg.GalleryStore(dim=dim, capacity=10000, device=local)
        st1.append_rows(G1, prenormalised=True)
        m1 = frg.Matcher(st1)
        for _ in range(20):
            r1 = m1.match(Q1, 1, 0.45, with_ids=False)
        t0 = time.perf_counter()
        for _ in range(200):
            r1 = m1.match(Q1, 1, 0.45, with_ids=False)
        gpu1_s = (time.perf_counter() - t0) / 200
        same1 = all((a[0] is None and r_ < 0) or (a[0] is not None and int(a[0], 16) == r_) for a, r_ in zip(res1, r1.rows[:, 0])) \
            and all(a[2] == bool(b) for a, b in zip(res1, r1.accept))
        st1.close()
        cpu = {"value": qps, "unit": UNIT, "cores": procs, "kind": "port",
               "config1_10k_x_64_one_core_queries_per_s": qps1,
               "config1_10k_x_64_gpu_e2e_queries_per_s": 64 / gpu1_s, "config1_gpu_ms_per_frame": gpu1_s * 1e3,
               "config1_gpu_agrees": bool(same1),
               "sample": "%d queries over %d worker processes x %d rows, top-1 + threshold 0.45, "
                         "per-face Python loop of peopleCount.py:860-887" % (q_cpu, procs, n),
               "seconds": per_step, "gpu_agrees": bool(same)}
        del G

    # ---- the other single-GPU configs of BASELINE.json, one parity-checked number each
    config3 = config5 = None
    if world == 1 and not args.bf16_only and not args.no_extra_configs and (n, dim) == (1_000_000, 512):
        config3 = run_config3(args, local, dev, peaks)
        config5 = run_config5(args, store, matcher, dev, n, dim)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if args.rows_total else "weak",
            "vs_baseline": None, "dtype": "f32" if variant == "scan_f32" else "bf16 filter + f32 rescore",
            "data": "synthetic", "config": workload_config(args, F, world), "variant": variant,
            "raw_queries_per_s": value / scale if sharded else value,
            "gallery_rows_total": n_total,
            "exchange": ({"path": smatcher.exchange,
                          "what": {"p2p": "frg_match_exchange: the select stage pushes each query's top-k to all ranks "
                                          "over NVLink peer memory as {payload, epoch} packets, a poll-only kernel merges "
                                          "(no collective call on the data path; bounded waits, status codes)",
                                   "nccl": "NCCL all_gather_into_tensor + frg_merge_topk_strided"}.get(
                                       smatcher.exchange, str(smatcher.exchange)),
                          "fallback_reason": smatcher.p2p_error,
                          "timeout_ms": int(os.environ["FRG_EXCHANGE_TIMEOUT_MS"])} if sharded else None),
            "config3": config3, "config4": config4, "config5": config5,
            "notes": ["e2e may exceed the device-timed value on a power-capped box: the per-step host synchronisation "
                      "of the e2e loop lets the SM clock recover between steps, the back-to-back device loop does not"],
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "pipelined": pipelined,
            "gpu_launches": main["launches_per_step"] * args.steps,
            "clocks": clocks, "parity": parity, "sweep": sweep, "peaks": peaks,
            "step_ms_spread": main["step_ms_spread"],
            "timing": "CUDA events on the launching stream around the K steps; only the dominant kernel is "
                      "bracketed inside the timed region, per-stage and per-step figures come from separate passes"}
    emit_json(line)


def timed_sharded_or_plain(step, steps, stream, dev, world):
    """CUDA events around `steps` calls of step(i); max over ranks."""
    import torch
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        step(i)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    return ms / steps


def run_config4(args, rank, world, local, dev, peaks):
    """BASELINE configs[3]: 512-d cosine, 100 M templates row-sharded over the ranks, batch 4096, top-10.
    Strong scaling: the gallery is fixed, raw queries/s is the figure.  Collective (every rank calls it)."""
    import torch
    import facerecognition_infrenceengine_b200 as frg
    from facerecognition_infrenceengine_b200 import _native as N
    from facerecognition_infrenceengine_b200.sharded import ShardedGallery, ShardedMatcher, shard_bounds
    from oracle import synth
    total, F, k, dim = args.config4_rows, args.config4_batch, 10, 512
    lo, hi = shard_bounds(total, world)[rank]
    rows = hi - lo
    # fp32 master + bf16 plane = 3 KB per row (2 GPUs: 154 GB each); fall back to the bf16-only store when
    # that does not fit beside what is already resident
    free_b, _ = torch.cuda.mem_get_info(dev)
    need = rows * (dim * 6 + 4) + (6 << 30)
    fits = torch.tensor([1 if free_b >= need else 0], device=dev)
    torch.distributed.all_reduce(fits, op=torch.distributed.ReduceOp.MIN)
    bf16_only = not bool(fits.item())
    store = frg.GalleryStore(dim=dim, capacity=rows, device=local, bf16_only=bf16_only)
    sg = ShardedGallery(dim=dim, device=local, store=store)
    sg.fill_synthetic(total, args.seed)
    sm = ShardedMatcher(sg, exchange=args.exchange)
    nb = 2
    QT = [synth.queries(F, total, dim, q0=i * F) for i in range(nb)]
    Qd = [torch.from_numpy(q).to(dev) for q, _ in QT]
    outs = [(torch.empty((F, k), dtype=torch.int64, device=dev), torch.empty((F, k), dtype=torch.float32, device=dev),
             torch.empty((F,), dtype=torch.uint8, device=dev)) for _ in range(nb)]
    stream = torch.cuda.current_stream(dev)

    def step(i):
        sm.match(Qd[i % nb], k, 0.45, variant=args.variant, out=outs[i % nb])

    torch.cuda.synchronize()
    torch.distributed.barrier()
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    launches = N.last_launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    per = timed_sharded_or_plain(step, 2, stream, dev, world)           # sizes the ~1 s of identical load
    pre = int(min(64, max(1, np.ceil(args.clock_preload_s / max(per * 1e-3, 1e-6)))))
    for i in range(pre):
        step(i)
    steps = max(20, args.steps)
    N.check(N.lib.frg_profile_enable(3))
    N.profile_collect()
    ms = timed_sharded_or_plain(step, steps, stream, dev, world)
    dom_ms, dom_launches = N.profile_collect()
    N.profile_enable(False)
    clocks = sampler.stop()
    sm.check_exchange()
    # ids verified on EVERY rank: the genuine queries' targets (known by construction, spread over all shards)
    # must come back first, lists ordered, no row twice
    ok = True
    for i in range(nb):
        r_, s_, a_ = (x.cpu().numpy() for x in outs[i])
        tgt = QT[i][1]
        hit = tgt >= 0
        ok &= bool((r_[hit, 0] == tgt[hit]).all()) and bool(a_[hit].all()) and not bool(a_[~hit].any())
        ok &= bool((np.diff(s_, axis=1) <= 0).all()) and all(len(set(x)) == k for x in r_[:64].tolist())
    t = torch.tensor([1.0 if ok else 0.0], device=dev)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MIN)
    pk = dict(peaks, use_sustained=power_capped(clocks))
    p_tc = pk["bf16_tflops_sustained"] if pk["use_sustained"] else pk["bf16_tflops"]
    t_roof = max(rows * dim * 2 / (pk["hbm_gbs"] * 1e9), 2.0 * F * rows * dim / (p_tc * 1e12)) * 1e3
    kern_ms = dom_ms / max(dom_launches, 1)
    out = {"workload": "configs[3]: 512-d cosine, %d-template gallery row-sharded over %d B200 (%d rows each), batch %d, "
                       "top-%d, peer-memory exchange + merge" % (total, world, rows, F, k),
           "scaling": "strong", "gallery_rows_total": total, "rows_per_gpu": rows, "batch": F, "k": k,
           "storage": "bf16-only plane (scores within eps[q] ~ 3.6e-3 of fp32)" if bf16_only else "fp32 master + bf16 scan plane",
           "exchange": sm.exchange, "steps": steps, "warmup": 3 + 2 + pre, "ms_per_step": ms,
           "value": F / (ms * 1e-3), "unit": UNIT, "launches_per_step": launches,
           "roofline_ms_per_step": t_roof, "roofline_queries_per_s": F / (t_roof * 1e-3),
           "step_frac_of_roofline": t_roof / ms,
           "kernel": {"name": "tc_scan_kernel<FILTER>", "launch_ms": kern_ms,
                      "achieved_tflops": 2.0 * F * rows * dim / (kern_ms * 1e-3) / 1e12 if kern_ms > 0 else None,
                      "peak_tflops": p_tc, "peak_kind": "sustained" if pk["use_sustained"] else "burst"},
           "ids_ok_all_ranks": bool(t.item() > 0), "clocks": clocks}
    del sm, sg
    store.close()
    return out


def run_config3(args, local, dev, peaks):
    """BASELINE configs[2]: 128-d Euclidean, 10 M gallery, batch 256, top-1 (our definition - the reference has
    no Euclidean path).  Tensor-core filter + exact rescoring, checked bit for bit against the exact fp32 scan."""
    import torch
    import facerecognition_infrenceengine_b200 as frg
    from facerecognition_infrenceengine_b200 import _native as N
    from oracle import matcher_oracle as mo
    from oracle import synth
    n, d, F, tol = args.config3_rows, 128, 256, 0.6
    store = frg.GalleryStore(dim=d, capacity=n, device=local, raw=True)
    store.fill_synthetic(n, 0, 99)
    m = frg.Matcher(store, metric="euclidean")
    Qh, tgt = synth.queries(F, n, d, seed=5, gallery_seed=99)
    Q = torch.from_numpy(Qh).to(dev)
    stream = torch.cuda.current_stream(dev)
    res = {}

    def step_v(variant):
        def step(i):
            res[variant] = m.match_device(Q, 1, tol, variant=variant, out=res.get(variant))
        return step

    for i in range(5):
        step_v("tc_exact")(i)
    N.check(N.lib.frg_profile_enable(3))
    N.profile_collect()
    ms = timed_sharded_or_plain(step_v("tc_exact"), max(20, args.steps), stream, dev, 1)
    dom_ms, dom_l = N.profile_collect()
    N.profile_enable(False)
    step_v("scan_f32")(0)
    torch.cuda.synchronize()
    tc = [t.cpu().numpy() for t in res["tc_exact"]]
    sc = [t.cpu().numpy() for t in res["scan_f32"]]
    same = bool(np.array_equal(tc[0], sc[0]) and np.array_equal(tc[1].view(np.uint32), sc[1].view(np.uint32))
                and np.array_equal(tc[2], sc[2]))
    # fp64 direct-difference oracle over the rows that can matter: every returned row and every target
    hit = tgt >= 0
    rows_chk = np.unique(np.concatenate([tc[0][:, 0], tgt[hit]]))
    Gs = synth.unit_rows(rows_chk, d, 99)
    ref_r, ref_d, ref_a = mo.euclidean_topk(Qh, Gs, 1, tol)
    oracle_ok = bool((rows_chk[ref_r[:, 0]] == tc[0][:, 0]).all() and np.abs(ref_d[:, 0] - tc[1][:, 0]).max() <= 1e-4
                     and (ref_a == tc[2].astype(bool)).all())
    roof = n * d * 4 / (peaks["hbm_gbs"] * 1e9) * 1e3
    out = {"workload": "configs[2]: 128-d Euclidean (ours; the reference has no Euclidean metric - parity unpinned), "
                       "%d-row gallery, batch %d, top-1" % (n, F),
           "gallery_rows": n, "dim": d, "batch": F, "k": 1, "ms_per_step": ms, "value": F / (ms * 1e-3), "unit": UNIT,
           "variant": "tc_exact (Euclidean scan plane)", "filter_kernel_ms": dom_ms / max(dom_l, 1),
           "roofline_ms_fp32_gallery_bytes": roof, "step_frac_of_roofline": roof / ms,
           "parity": {"bit_identical_to_exact_scan": same, "genuine_found": bool((tc[0][hit, 0] == tgt[hit]).all()),
                      "fp64_oracle_on_returned_and_target_rows_ok": oracle_ok, "tolerance": 1e-4}}
    store.close()
    return out


def run_config5(args, store, matcher, dev, n, dim):
    """BASELINE configs[4]: peopleCount video stream - 32 frames x up to 50 faces = 1600 faces per batch against the
    1 M gallery, with online enrol / evict between batches (64 upserts + 16 removals, host buffers).  Runs last: it
    mutates the store."""
    import torch
    from oracle import synth
    F, steps, warm = 1600, max(20, args.steps), 5
    Qh, tgt = synth.queries(F, n, dim, q0=900_000)
    Q = torch.from_numpy(Qh).to(dev)
    new = synth.unit_rows(np.arange(64 * (steps + warm)), dim, 777, synth.STREAM_IMPOSTOR).reshape(steps + warm, 64, dim)
    res = None
    stream = torch.cuda.current_stream(dev)

    def match_only(i):
        nonlocal res
        res = matcher.match_device(Q, 1, 0.45, variant=args.variant, out=res)

    def step(i):
        match_only(i)
        store.upsert(["new%d_%d" % (i, j) for j in range(64)], new[i])           # 64 enrolments per batch
        if i:
            store.remove(["new%d_%d" % (i - 1, j) for j in range(0, 64, 4)])      # 16 evictions per batch

    for i in range(warm):
        step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(warm, warm + steps):
        step(i)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    match_ms = timed_sharded_or_plain(match_only, steps, stream, dev, 1)
    last = warm + steps - 1
    probe = np.stack([new[last][1], new[last - 1][0], new[last - 1][1]])      # fresh, evicted, kept
    r = matcher.match(probe, 1, 0.45)
    rows = res[0].cpu().numpy()
    hit = tgt >= 0
    return {"workload": "configs[4]: 32 frames x 50 faces = %d faces per batch against the %d-row gallery, 64 enrolments + "
                        "16 evictions (host buffers) between batches" % (F, n),
            "batch": F, "k": 1, "steps": steps, "ms_per_step_with_updates": dt * 1e3, "value": F / dt, "unit": UNIT,
            "ms_per_step_match_only": match_ms, "queries_per_s_match_only": F / (match_ms * 1e-3),
            "timing": "wall clock around match + upsert + remove calls (mutators are asynchronous host calls)",
            "parity": {"fresh_rows_found": bool(r.accept[0] and r.accept[2] and r.ids[0][0] == "new%d_1" % last),
                       "evicted_row_rejected": bool(not r.accept[1]),
                       "genuine_found": bool((rows[hit, 0] == tgt[hit]).all())}}


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries write banners to stdout (NCCL: "NCCL version ..." at communicator creation).  The contract is
    ONE JSON line on stdout: point fd 1 at stderr for the whole run and keep the real stdout for emit_json()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


DUMP_LIMIT_BYTES = 60 << 20          # data bytes: the files stay under 64 MB (10^6 or 2^20) with their headers


def dump_outputs(path, rows, scores, accept):
    """--dump-outputs: what the last timed step handed its caller, one DIR/<name>.npy per array, so that two
    builds run with the same arguments (hence the same inputs) can be compared output for output.

      rows.npy         float64 [F, k]  gallery rows, best first (-1: no row)
      scores.npy       float32 [F, k]
      accept.npy       float32 [F]     1 = the best score reaches the threshold
      query_index.npy  float64 [F]     position of each written query in the batch

    Where the whole batch would pass DUMP_LIMIT_BYTES, a fixed seeded sample of the queries is written, in batch
    order."""
    F = len(rows)
    per_query = rows.shape[1] * (8 + 4) + 4 + 8
    keep = np.arange(F)
    if F * per_query > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(F, DUMP_LIMIT_BYTES // per_query, replace=False))
    os.makedirs(path, exist_ok=True)
    for name, a in (("rows", rows[keep].astype(np.float64)), ("scores", scores[keep].astype(np.float32)),
                    ("accept", accept[keep].astype(np.float32)), ("query_index", keep.astype(np.float64))):
        np.save(os.path.join(path, name + ".npy"), a)


def ncu_traffic(variant, n, dim, F, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the ncu --set full
    capture committed under profiles/ (only when it was taken on this very workload), else None."""
    if world != 1 or variant != "tc_exact" or (n, dim) != (1_000_000, 512):
        return None, None
    name = {1024: "r02_ncu_full_tc_scan_b1024_grouped.txt", 64: "r01_ncu_full_tc_scan_b64_v1.txt"}.get(F)
    path = os.path.join(ROOT, "profiles", name) if name else None
    if not path or not os.path.exists(path):
        return None, None
    rd = wr = None
    in_filter = False
    scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
    for line in open(path):
        if line.startswith("== "):
            in_filter = "tc_scan_kernel<1" in line
        elif in_filter and "dram__bytes_read.sum" in line:
            f = line.split()
            rd = float(f[1]) * scale[f[2]]
        elif in_filter and "dram__bytes_write.sum" in line:
            f = line.split()
            wr = float(f[1]) * scale[f[2]]
    if rd is None or wr is None:
        return None, None
    return rd + wr, "profiles/" + name


def step_roofline_ms(n, dim, F, peaks, bytes_per_elem=2):
    """Whole-step roofline: the slower of the scan-plane bytes at HBM speed and 2*F*n*dim flops at the
    tensor peak (sustained figure when the run was power-capped)."""
    p_tc = peaks["bf16_tflops_sustained"] if peaks.get("use_sustained") else peaks["bf16_tflops"]
    return max(n * dim * bytes_per_elem / (peaks["hbm_gbs"] * 1e9), 2.0 * F * n * dim / (p_tc * 1e12)) * 1e3


def tc_roofline(variant, n, dim, F, launch_ms, peaks):
    flops = 2.0 * F * n * dim
    bytes_ = n * dim * 2
    t_hbm = bytes_ / (peaks["hbm_gbs"] * 1e9)
    # B200_PROFILING.md: burst cuBLAS figure for a kernel timed alone, sustained one for a kernel inside a
    # long power-capped run - which is the regime here whenever the clock record shows sw_power_cap
    sustained = bool(peaks.get("use_sustained"))
    p_tc = peaks["bf16_tflops_sustained"] if sustained else peaks["bf16_tflops"]
    t_tc = flops / (p_tc * 1e12)
    if t_tc >= t_hbm:
        ach = flops / (launch_ms * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": "tc_scan_kernel<FILTER>", "achieved": ach, "peak": p_tc,
                "peak_kind": "sustained (sw_power_cap active during the run)" if sustained else "burst",
                "frac_of_burst_peak": ach / peaks["bf16_tflops"],
                "unit": "TFLOP/s", "frac": ach / p_tc, "traffic": None,
                "algorithmic_flops_per_launch": flops, "launch_ms": launch_ms, "peak_source": peaks["source"]}
    ach = bytes_ / (launch_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "tc_scan_kernel<FILTER>", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": ach / peaks["hbm_gbs"], "traffic": None, "algorithmic_bytes_per_launch": bytes_,
            "launch_ms": launch_ms, "peak_source": peaks["source"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--variant", default="auto")
    ap.add_argument("--sweep", default="1,8,64,128,256,512,1024")
    ap.add_argument("--bf16-only", action="store_true",
                    help="bf16 gallery mode: only the bf16 scan plane is resident (1 KB / row); scores within ~3.6e-3 (7.9e-3 worst case)")
    ap.add_argument("--clock-preload-s", type=float, default=1.0,
                    help="seconds of untimed identical load before the timed region, for the clock sampler")
    ap.add_argument("--rows-total", type=int, default=0,
                    help="fixed total gallery, row-sharded over the ranks (BASELINE configs[3]: 100000000 with "
                         "--batch 4096 --k 10); default: --rows per GPU")
    ap.add_argument("--shard", default="gallery", choices=["gallery", "queries"],
                    help="N>1: row-shard the gallery (all-gather + merge) or replicate it and shard the query stream")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"],
                    help="N>1, row-sharded: pushes from the match kernels + a poll-and-merge kernel over NVLink peer memory, or NCCL "
                         "all-gather + merge kernel; auto = p2p when the peer mapping can be set up")
    ap.add_argument("--e2e-callers", type=int, default=2,
                    help="host threads of the extra concurrent end-to-end measurement (1 = skip it)")
    ap.add_argument("--config4-rows", type=int, default=100_000_000,
                    help="N>1: total rows of the fixed-gallery leg (BASELINE configs[3]); 0 = skip it")
    ap.add_argument("--config4-batch", type=int, default=4096)
    ap.add_argument("--config3-rows", type=int, default=10_000_000)
    ap.add_argument("--no-extra-configs", action="store_true", help="N=1: skip the config 3 / config 5 legs")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--cpu-procs", type=int, default=0)
    ap.add_argument("--cpu-queries", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rows, scores and accept decisions of the last timed step as DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    quiet_stdout()
    if args.impl == "reference":
        reference_arm(args, rank, world)
    else:
        try:
            ours_arm(args, rank, world)
        finally:
            if world > 1:
                import torch.distributed as dist
                if dist.is_initialized():
                    dist.destroy_process_group()


if __name__ == "__main__":
    main()
