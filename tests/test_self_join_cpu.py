"""The numpy reference of the gallery self-join against the range oracle it is built on: every pair a < b of the
range search over all rows, with the tag rule applied afterwards, and nothing else."""
import numpy as np
import pytest

from oracle import matcher_oracle as mo
from oracle import synth
from range_oracle import range_search
from self_join_oracle import self_join_reference


def _gallery(n=300, d=128, seed=5):
    rng = np.random.default_rng(seed)
    G = synth.gallery(n, d, seed)
    for a, b in rng.choice(n, (20, 2), replace=False):
        G[b] = mo.normalise(G[a] + 0.2 * synth.gallery(1, d, int(b) + 7)[0])
    G[17] = G[3]                                    # an exact copy
    with np.errstate(invalid="ignore", divide="ignore"):
        G[40] = np.zeros(d, np.float32) / np.float32(0)   # a zero row stored as NaN
    tags = rng.integers(0, 4, n).astype(np.int32)
    tags[rng.choice(n, 15, replace=False)] = -1     # tombstones
    tags[3] = tags[17] = 1                          # the copy and its source: live, one company
    return G, tags


@pytest.mark.parametrize("tenant,same_tag,strict", [(-1, False, False), (-1, True, True), (2, False, True),
                                                    (2, True, False)])
def test_reference_is_the_range_oracle_upper_triangle(tenant, same_tag, strict):
    G, tags = _gallery()
    thr = 0.25
    counts, rows, scores = self_join_reference(G, tags, thr, tenant, same_tag, strict)
    live = tags >= 0
    _, all_r, all_s = range_search(G, G, thr, mask=live, strict=strict)
    for a in range(len(G)):
        ok_a = tags[a] >= 0 and (tenant < 0 or tags[a] == tenant)
        keep = [(int(b), float(s)) for b, s in zip(all_r[a], all_s[a])
                if ok_a and b > a and (tenant < 0 or tags[b] == tenant) and (not same_tag or tags[b] == tags[a])]
        keep.sort()
        assert counts[a] == len(keep)
        assert rows[a].tolist() == [b for b, _ in keep]
        # one query against the gallery vs a batch of queries: BLAS may round the last bit differently
        assert np.allclose(scores[a], np.array([s for _, s in keep], np.float32), rtol=0, atol=2e-6)
    assert counts[3] >= 1 or (tenant >= 0 and tenant != 1)
    assert counts[40] == 0                          # a NaN row matches nothing


def test_reference_subset_of_rows():
    G, tags = _gallery(n=200)
    full = self_join_reference(G, tags, 0.2)
    some = np.array([0, 5, 199, 77])
    part = self_join_reference(G, tags, 0.2, rows=some)
    assert np.array_equal(part[0], full[0][some])
    for i, a in enumerate(some):
        assert np.array_equal(part[1][i], full[1][a]) and np.array_equal(part[2][i], full[2][a])
