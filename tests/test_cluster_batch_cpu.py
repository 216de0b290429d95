"""Batched unknown-face clustering without a device: the premises frg_cluster_observe_host is built on.
  (i)  np.mean(window, axis=0) of fp32 rows == a sequential fp32 sum from +0.0f, oldest first, then one fp32 division
       (the resolve kernel's mean), bit for bit;
  (ii) the two-phase algorithm (pre-pass with a hit budget of 16, touched set, truncated-list rescan) gives what
       UnknownClusterOracle.observe gives face by face: clusters, created flags and means."""
import copy

import numpy as np
import pytest

from cluster_streams import branch_streams, np_mean, people_stream, two_phase
from oracle.matcher_oracle import UnknownClusterOracle


def device_mean(window: np.ndarray) -> np.ndarray:
    s = np.zeros(window.shape[1], np.float32)
    for row in window:
        s = (s + row).astype(np.float32)
    return (s / np.float32(len(window))).astype(np.float32)


@pytest.mark.parametrize("n", range(1, 17))
def test_mean_is_sequential_fp32_sum_then_division(n):
    rng = np.random.default_rng(n)
    for trial in range(40):
        W = (rng.standard_normal((n, 64)) * 10.0 ** rng.integers(-3, 3)).astype(np.float32)
        W[rng.random(W.shape) < 0.1] = -0.0
        if trial % 5 == 0:
            W[:, :8] = -0.0                                   # whole columns of -0.0: the sum starts from +0.0f
        ref = np_mean(list(W))
        assert ref.dtype == np.float32
        got = device_mean(W)
        assert np.array_equal(ref.view(np.uint32), got.view(np.uint32))


def test_mean_of_negative_zeros_is_positive_zero():
    for n in (1, 2, 10):
        m = np_mean([np.full(4, -0.0, np.float32)] * n)
        assert not np.signbit(m).any()


def _oracle_after(before, threshold=0.65, window=10):
    o = UnknownClusterOracle(threshold=threshold, window=window)
    for q in before:
        o.observe(q)
    return o


def _check(before, batch, threshold=0.65, window=10):
    o = _oracle_after(before, threshold, window)
    avg, members = copy.deepcopy(o.avg), copy.deepcopy(o.members)
    stats = {}
    got = two_phase(avg, members, batch, threshold, window=window, stats=stats)
    want = [o.observe(q) for q in batch]
    assert got == want
    assert len(avg) == len(o.avg)
    for a, b in zip(avg, o.avg):
        assert np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))
    assert [list(map(bytes, d)) for d in members] == [list(map(bytes, d)) for d in o.members]
    return stats


def test_two_phase_takes_every_branch():
    before, batch = branch_streams(64)
    stats = _check(before, batch)
    assert stats.get("rescan", 0) >= 1                    # 16 listed hits touched, list truncated
    assert stats.get("first_hit_touched", 0) >= 2         # recomputed hits, one of which no longer qualifies
    assert stats.get("join_new", 0) >= 2                  # joins of a cluster founded in the batch
    o = _oracle_after(before)
    res = [o.observe(q) for q in batch]
    assert res[1] == (21, True)                           # the moved mean no longer takes the face it took before
    assert res[2] == (20, False)
    assert res[19] == (16, False)                         # found by the rescan past the 16 listed hits


@pytest.mark.parametrize("seed", range(6))
def test_two_phase_equals_sequential_on_random_streams(seed):
    rng = np.random.default_rng(seed)
    dim = 64
    Q = people_stream(rng, dim, people=int(rng.integers(3, 25)), n=300, noise=float(rng.uniform(0.6, 0.9)))
    if seed % 2:
        Q[rng.integers(0, len(Q), 3)] = np.nan                # normalised zero faces
    cut = int(rng.integers(0, 120))
    stats = _check(Q[:cut], Q[cut:], window=int(rng.integers(1, 17)))
    assert stats.get("first_hit_touched", 0) > 0


def test_two_phase_window_wraps_and_many_hits():
    rng = np.random.default_rng(7)
    dim = 64
    # 40 clusters, all hit by one direction; a batch that joins them repeatedly (windows wrap) and probes them
    a, b = 0.75, float(np.sqrt(1 - 0.75 ** 2))
    before = [((a * np.eye(dim)[0] + b * np.eye(dim)[k + 1])).astype(np.float32) for k in range(40)]
    batch = []
    for _ in range(30):
        k = int(rng.integers(0, 40))
        batch.append((before[k] + 0.05 * rng.standard_normal(dim)).astype(np.float32))
        if rng.random() < 0.3:
            batch.append(np.eye(dim, dtype=np.float32)[0])
    _check(before, np.stack(batch), window=3)
