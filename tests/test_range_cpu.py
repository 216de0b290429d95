"""Range search, host side without a GPU: the numpy reference against the top-k oracle, and the collective
``ShardedMatcher.match_range`` over world-size-2 `gloo` processes with the per-shard range search injected from the
reference (concatenation in rank order, truncation, the retry decided from the gathered counts)."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import matcher_oracle as mo
from oracle import synth
from range_oracle import range_search


@pytest.mark.parametrize("k", [1, 4, 16])
@pytest.mark.parametrize("masked", [False, True])
def test_range_prefix_is_topk(k, masked):
    rng = np.random.default_rng(k + 7 * masked)
    n, d = 3000, 128
    G = synth.gallery(n, d, 11)
    G[17] = G[5]                                                    # an exact tie: lower row first
    G[40] = np.nan
    Q = np.concatenate([G[[5, 99]], rng.standard_normal((6, d)).astype(np.float32)])
    tags = rng.integers(-1, 3, n).astype(np.int32) if masked else None
    mask = None if tags is None else tags >= 0
    counts, rows, scores = range_search(Q, G, -1.0, mask=mask, strict=True)        # every row above -1
    ref_r, ref_s, _ = mo.match_topk_fast(Q, G, k, 0.4, tags=tags)
    for f in range(len(Q)):
        m = min(k, counts[f])
        assert np.array_equal(rows[f][:m], ref_r[f, :m]) and np.array_equal(scores[f][:m], ref_s[f, :m])
        assert (ref_r[f, m:] == -1).all()
    # the threshold rule itself: >= by default, > when strict, on the fp32 scores
    thr = float(mo.cosine_scores(Q[:1], G)[0, 5])          # (a 1-row product may round differently from a batch)
    c_ge, r_ge, _ = range_search(Q[:1], G, thr)
    c_gt, r_gt, _ = range_search(Q[:1], G, thr, strict=True)
    assert 5 in r_ge[0] and 17 in r_ge[0] and 5 not in r_gt[0] and c_ge[0] == c_gt[0] + 2


def test_range_euclidean_rule():
    G = np.array([[0, 0], [3, 4], [6, 8], [np.nan, 0]], np.float32)
    counts, rows, scores = range_search(np.zeros((1, 2), np.float32), G, 5.0, metric="euclidean")
    assert counts[0] == 2 and list(rows[0]) == [0, 1] and list(scores[0]) == [0.0, 5.0]
    counts, rows, _ = range_search(np.zeros((1, 2), np.float32), G, 5.0, metric="euclidean", strict=True)
    assert counts[0] == 1 and list(rows[0]) == [0]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from facerecognition_infrenceengine_b200.sharded import ShardedGallery, ShardedMatcher
        n, d = 4001, 128
        G = synth.gallery(n, d, 3)
        G[3000:3040] = G[10]                         # 41 copies of row 10, most of them on rank 1
        tags = np.where(np.arange(n) % 3 == 0, -1, 1).astype(np.int32)      # tombstones
        Q = np.concatenate([G[[10, 20]], synth.gallery(3, d, 4)])
        g = ShardedGallery(dim=d, store=None)
        lo, hi = g.plan(n)
        calls = []

        def local_range(Qx, thr, strict, tenant, max_hits, row_offset):
            calls.append((len(Qx), max_hits))
            counts, rows, scores = range_search(Qx, G[lo:hi], thr, mask=tags[lo:hi] >= 0, strict=strict)
            out_r = np.full((len(Qx), max_hits), -1, np.int64)
            out_s = np.full((len(Qx), max_hits), -1.0, np.float32)
            for f in range(len(Qx)):
                order = np.argsort(rows[f], kind="stable")[:max_hits]          # gallery order, as the C layer
                out_r[f, :len(order)] = rows[f][order] + row_offset
                out_s[f, :len(order)] = scores[f][order]
            return counts, out_r, out_s

        m = ShardedMatcher(g, local_match=lambda *a, **k: None, merge=lambda *a, **k: None)
        res = m.match_range(Q, 0.3, max_hits=4, with_ids=False, local_range=local_range)
        ref_c, ref_r, ref_s = range_search(Q, G, 0.3, mask=tags >= 0)
        assert np.array_equal(res.counts, ref_c), (res.counts, ref_c)
        for f in range(len(Q)):
            # (the shards' products round by an ulp differently from the whole gallery's: ranks of equal scores
            # are compared as sets)
            assert sorted(res.rows[f]) == sorted(ref_r[f]) and np.abs(np.sort(res.scores[f]) - np.sort(ref_s[f])).max(initial=0) < 1e-6, f
            assert (np.diff(res.scores[f]) <= 0).all()
        assert ref_c[0] > 4 and ref_c.min() <= 4
        # one first call, then ONE retry of the truncated queries only, sized by their largest TOTAL count
        assert calls == [(len(Q), 4), (int((ref_c > 4).sum()), int(ref_c.max()))], calls
        ret[rank] = 1
    finally:
        dist.destroy_process_group()


def test_sharded_range_world2_gloo():
    import facerecognition_infrenceengine_b200  # noqa: F401  (builds / loads the library before forking)
    port = _free_port()
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=180)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    assert dict(ret) == {0: 1, 1: 1}
