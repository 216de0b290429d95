"""CPU rehearsal of the int8 cosine filter's error band (numpy only, no GPU).

For the synthetic gallery (oracle/synth) and a slice of the benchmark queries it quantises both sides the way the
device does (gallery: step alpha / 127, alpha = 0.165 at dim 512; query: step max|q| / 127), computes eps[q] with the
prep kernel's formula, and reports per query (median / p99 / max):
  - dense candidates of the filter for the exact sample floor e_k - eps (k best group winners of the pre-pass sample,
    rescored exactly) at pre-pass strides 8 / 16 / 32, and for the group-maximum floor L - 2 eps;
  - rows the select stage rescores (coarse >= tau_e - eps) against its 256-row budget;
  - range candidates at threshold 0.15 (floor 0.15 - eps) against the 4096-entry budget.
It asserts that every true top-k row survives every band.

    python tools/int8_band_sim.py [--rows 1000000] [--queries 128] [--k 5] [--alpha 0.165] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from oracle import synth  # noqa: E402

TILE = 256          # rows per pre-pass tile of the CTA-pair filter (1024 queries)
GROUPS = 32


def quant(x, step):
    return np.clip(np.rint(x / step), -127, 127)


def stats(v):
    v = np.asarray(v)
    return [int(np.median(v)), int(np.percentile(v, 99)), int(v.max())]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--queries", type=int, default=128)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--alpha", type=float, default=0.0, help="gallery scale (0: 0.165 * sqrt(512 / dim))")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    n, d, k = a.rows, a.dim, a.k
    alpha = a.alpha or 0.165 * np.sqrt(512.0 / d)
    G = synth.gallery(n, d)
    Q, _ = synth.queries(1024, n, d)
    Q = Q[:a.queries]
    Q = (Q / np.linalg.norm(Q, axis=1, keepdims=True)).astype(np.float32)
    cg = np.float32(alpha / 127)
    Gi = quant(G, cg).astype(np.float32)
    rg = float(((G - Gi * cg) ** 2).sum(1).max())
    cq = (np.abs(Q).max(1) / 127).astype(np.float32)
    Qi = quant(Q, cq[:, None]).astype(np.float32)
    rq = ((Q - Qi * cq[:, None]) ** 2).sum(1)
    eps = 1.01 * ((1 + np.sqrt(rq)) * np.sqrt(rg) + np.sqrt(rq)) + 4e-5
    S = (Qi @ Gi.T) * (cq[:, None] * cg)                  # integer products are exact in fp32 (< 2^24)
    E = Q @ G.T
    top = np.argsort(-E, axis=1, kind="stable")[:, :k]
    tau = np.take_along_axis(E, top[:, -1:], 1)[:, 0]
    out = {"rows": n, "dim": d, "queries": len(Q), "k": k, "alpha": alpha, "saturated_elements": int((np.abs(G) > alpha).sum()),
           "eps_median": float(np.median(eps)), "eps_max": float(eps.max()), "floors": {}}
    rows = np.arange(n)
    for stride in (8, 16, 32):
        sample = (rows // TILE) % stride == 0
        gidx = [np.nonzero(sample & (rows % GROUPS == g))[0] for g in range(GROUPS)]
        dense_exact, dense_gmax = [], []
        for f in range(len(Q)):
            gbest = np.full(GROUPS, -np.inf)
            grow = np.zeros(GROUPS, np.int64)
            for g, idx in enumerate(gidx):
                j = idx[np.argmax(S[f, idx])]
                gbest[g], grow[g] = S[f, j], j
            order = np.argsort(-gbest)[:k]
            e_k = E[f, grow[order]].min()
            fl_exact = e_k - eps[f]
            fl_gmax = np.sort(gbest)[-k] - 2 * eps[f]
            assert (S[f, top[f]] >= fl_exact).all() and (S[f, top[f]] >= fl_gmax).all(), (stride, f)
            dense_exact.append(int((S[f] >= fl_exact).sum()))
            dense_gmax.append(int((S[f] >= fl_gmax).sum()))
        out["floors"][str(stride)] = {"exact_sample_floor": stats(dense_exact), "group_max_floor": stats(dense_gmax),
                                      "stage_entries": int(min(8192, max(256, 3.0 * stride * (k + 10 * np.sqrt(k) + 10))))}
    # select: tau_e from the k best coarse rows, keep coarse >= tau_e - eps
    coarse_top = np.argsort(-S, axis=1, kind="stable")[:, :k]
    tau_e = np.take_along_axis(E, coarse_top, 1).min(1)
    keep = (S >= (tau_e - eps)[:, None]).sum(1)
    assert (np.take_along_axis(S, top, 1) >= (tau_e - eps)[:, None]).all()
    assert (tau_e <= tau).all()
    out["select_rescored"] = stats(keep) + [256]
    rng = (S >= (0.15 - eps)[:, None]).sum(1)
    assert ((S >= (0.15 - eps)[:, None]) | (E < 0.15)).all()
    out["range_0p15_candidates"] = stats(rng) + [4096]
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
