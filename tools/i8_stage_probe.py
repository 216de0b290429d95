"""Per-stage device times of the int8 top-k path at the headline shape (1 M x 512 unit gallery, top-5) and batch sizes
64 / 256 / 1024: query prep, int8 pre-pass, floor, filter, select + rescore and the exact fallback, each bracketed by
CUDA events.  Every batch size first runs the identical call for >= --preload-s seconds, so the card sits at the clock
it holds under this load; the SM clock is sampled (nvidia-smi query only) while the timed calls run.

The filter's time is also given per tile and SM (pair) in clocks at the sampled clock, beside the tensor pipe's floor
for that tile: 2 * M * N * dim int8 operations at 16384 per clock and SM (M = N = 128 per CTA, 256 across a pair).

    python tools/i8_stage_probe.py [--batches 64,256,1024] [--steps 50] [--label NAME] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import facerecognition_infrenceengine_b200 as frg  # noqa: E402
from facerecognition_infrenceengine_b200 import _native as N  # noqa: E402
from oracle import synth  # noqa: E402

I8_OPS_PER_CLK_SM = 16384


def smi_id():
    """nvidia-smi's name for the card torch runs on (its PCI bus id: device 0 of the process need not be nvidia-smi's
    device 0 under CUDA_VISIBLE_DEVICES)."""
    pr = torch.cuda.get_device_properties(torch.cuda.current_device())
    return "%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)


def smi(fields):
    return subprocess.run(["nvidia-smi", "-i", smi_id(), "--query-gpu=" + fields, "--format=csv,noheader,nounits"],
                          capture_output=True, text=True).stdout.strip()


class ClockSampler:
    def __init__(self):
        self.vals, self.proc = [], None

    def __enter__(self):
        self.proc = subprocess.Popen(["nvidia-smi", "-i", smi_id(), "--query-gpu=clocks.sm", "--format=csv,noheader,nounits",
                                      "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        self.t = threading.Thread(target=self._pump, daemon=True)
        self.t.start()
        return self

    def _pump(self):
        for line in self.proc.stdout:
            try:
                self.vals.append(float(line.strip()))
            except ValueError:
                pass

    def __exit__(self, *exc):
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        self.t.join(timeout=5)

    def median(self):
        return statistics.median(self.vals) if self.vals else None


def tile_shape(F, rows, sm_count):
    """(tiles per SM or SM pair, tensor-pipe clocks per tile) of the filter launch, as tc_plan lays it out."""
    qtiles = (F + 127) // 128
    pair = qtiles >= 2
    if pair:
        qtiles += qtiles & 1
        cols, units, tile_rows = qtiles // 2, sm_count // 2, 256
    else:
        cols, units, tile_rows = qtiles, sm_count, 128
    tiles = (rows + tile_rows - 1) // tile_rows
    m = 256 if pair else 128
    clk = 2 * m * tile_rows * 512 / (I8_OPS_PER_CLK_SM * (2 if pair else 1))
    return cols * tiles / units, clk


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--batches", default="64,256,1024")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--preload-s", type=float, default=1.0)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    d, k = 512, 5
    card = smi("name,power.limit,clocks.max.sm,pci.bus_id").split(", ")
    assert len(card) == 4, "nvidia-smi does not know the card at %s" % smi_id()
    sm_count = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    store = frg.GalleryStore(dim=d, capacity=a.rows)
    store.fill_synthetic(a.rows, 0, synth.GALLERY_SEED)
    m = frg.Matcher(store)
    Qall = torch.from_numpy(synth.queries(max(int(x) for x in a.batches.split(",")), a.rows, d)[0]).cuda()
    res = {"label": a.label, "gpu": card[0], "power_limit_w": float(card[1]), "sm_max_mhz": float(card[2]), "pci_bus_id": card[3],
           "rows": a.rows, "dim": d, "k": k, "steps": a.steps, "preload_s": a.preload_s, "batches": {}}
    for F in [int(x) for x in a.batches.split(",")]:
        Q = Qall[:F].contiguous()
        out = m.match_device(Q, k, frg.CAMPUS_THRESHOLD)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < a.preload_s:
            for _ in range(10):
                m.match_device(Q, k, frg.CAMPUS_THRESHOLD, out=out)
            torch.cuda.synchronize()
        with ClockSampler() as clocks:
            # whole steps without the per-stage events first, then the same calls with them
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                m.match_device(Q, k, frg.CAMPUS_THRESHOLD, out=out)
            e1.record()
            torch.cuda.synchronize()
            N.profile_enable(True)
            N.profile_collect()
            for _ in range(a.steps):
                m.match_device(Q, k, frg.CAMPUS_THRESHOLD, out=out)
            torch.cuda.synchronize()
            N.profile_collect()
            st = {name: v / a.steps * 1e3 for name, v in N.profile_stages().items()}
            N.profile_enable(False)
        mhz = clocks.median()
        tiles, floor_clk = tile_shape(F, a.rows, sm_count)
        filt_clk = st["dominant"] * 1e-6 * mhz * 1e6 / tiles if mhz else None
        row = {"step_us": e0.elapsed_time(e1) / a.steps * 1e3, "variant": N.last_variant(),
               "stage_us": {("filter" if n == "dominant" else n): round(v, 2) for n, v in st.items()},
               "sm_mhz_median": mhz, "tiles_per_unit": round(tiles, 1), "mma_floor_clk_per_tile": floor_clk,
               "filter_clk_per_tile": round(filt_clk, 1) if filt_clk else None,
               "filter_over_mma_floor": round(filt_clk / floor_clk, 3) if filt_clk else None}
        res["batches"][str(F)] = row
        print(F, json.dumps(row), flush=True)
    store.close()
    txt = json.dumps(res, indent=1)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
