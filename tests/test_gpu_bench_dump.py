"""bench.py --dump-outputs on a small gallery: the files hold what the last timed step returned to its caller."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import matcher_oracle as mo
from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_last_timed_step(tmp_path):
    n, dim, F, k, steps = 20000, 512, 64, 5, 7
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(n), "--dim", str(dim),
                        "--batch", str(F), "--k", str(k), "--steps", str(steps), "--warmup", "2", "--sweep", "",
                        "--no-cpu", "--no-extra-configs", "--e2e-callers", "1", "--clock-preload-s", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    out = {name: np.load(tmp_path / (name + ".npy")) for name in ("rows", "scores", "accept", "query_index")}
    assert out["rows"].dtype == np.float64 and out["scores"].dtype == np.float32
    assert out["accept"].dtype == np.float32 and out["query_index"].dtype == np.float64
    assert out["rows"].shape == (F, k) and np.array_equal(out["query_index"], np.arange(F))
    # bench.py cycles through four query batches: step i matches batch i % 4
    Q, _ = synth.queries(F, n, dim, q0=((steps - 1) % 4) * F)
    ref_rows, ref_scores, ref_acc = mo.match_topk(Q, synth.gallery(n, dim), k + 1, 0.45)
    assert mo.ids_match_with_gap(ref_rows, ref_scores, out["rows"].astype(np.int64), 1e-4).all()
    assert np.abs(out["scores"] - ref_scores[:, :k]).max() <= 1e-4
    assert (out["accept"].astype(bool) == ref_acc).all()
