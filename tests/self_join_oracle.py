"""Numpy reference of the gallery self-join (test infrastructure): tests/range_oracle.py restricted to the upper
triangle.  Row a's stored vector is the query; row b counts for it when b > a, b is live, and the tag rule holds."""
from typing import Optional

import numpy as np

from range_oracle import range_search


def self_join_reference(G: np.ndarray, tags: np.ndarray, threshold: float, tenant: int = -1, same_tag: bool = False,
                        strict: bool = False, rows: Optional[np.ndarray] = None):
    """(counts int64[len(rows)], per-row hit rows in GALLERY order, their scores) for the query rows `rows` (default:
    all).  A dead query row, or one outside `tenant`, has no hits."""
    G = np.asarray(G, np.float32)
    tags = np.asarray(tags, np.int32)
    idx = np.arange(len(G))
    rows = idx if rows is None else np.asarray(rows)
    counts = np.zeros(len(rows), np.int64)
    out_r, out_s = [], []
    for i, a in enumerate(rows.tolist()):
        ta = int(tags[a])
        mask = (tags >= 0) & (idx > a)
        if tenant >= 0:
            mask &= tags == tenant
        if same_tag:
            mask &= tags == ta
        if ta < 0 or (tenant >= 0 and ta != tenant):
            mask &= False
        c, r, s = range_search(G[a:a + 1], G, threshold, mask=mask, strict=strict)
        order = np.argsort(r[0], kind="stable")
        counts[i] = c[0]
        out_r.append(r[0][order])
        out_s.append(s[0][order])
    return counts, out_r, out_s
