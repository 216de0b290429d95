"""Numpy reference of the range search (test infrastructure, beside oracle/matcher_oracle.py whose conventions it
follows: fp32 scores of normalise(q) . g, NaN never qualifies, ties by gallery row)."""
from typing import List, Optional

import numpy as np

from oracle.matcher_oracle import cosine_scores


def range_search(Q: np.ndarray, G: np.ndarray, threshold: float, mask: Optional[np.ndarray] = None,
                 strict: bool = False, metric: str = "cosine", chunk: int = 128):
    """Range search (OUR extension - parity unpinned, like k > 1 and Euclidean): every row whose score reaches the
    threshold.  Cosine: fp32 ``normalise(q) . g >= threshold`` ('>' when strict); Euclidean: ``||g - q|| <= threshold``
    ('<' when strict), direct difference as :func:`euclidean_topk`.  NaN never qualifies; ``mask`` bool[N] selects
    the rows that take part.  Returns (counts int64[F], rows, scores): per query the COMPLETE lists, best first
    (score desc / distance asc, then row asc) - so its first k entries are :func:`match_topk_fast`'s."""
    Q = np.asarray(Q, dtype=np.float32)
    G = np.asarray(G, dtype=np.float32)
    F = len(Q)
    thr = np.float32(threshold)
    counts = np.zeros(F, np.int64)
    rows: List[np.ndarray] = []
    scores: List[np.ndarray] = []
    for a in range(0, F, chunk):
        if metric == "cosine":
            S = cosine_scores(Q[a:a + chunk], G) if len(G) else np.zeros((len(Q[a:a + chunk]), 0), np.float32)
            ok = (S > thr) if strict else (S >= thr)
        else:
            S = np.stack([np.sqrt(np.sum((G.astype(np.float64) - q.astype(np.float64)) ** 2, axis=1)).astype(np.float32)
                          for q in Q[a:a + chunk]]) if len(G) else np.zeros((len(Q[a:a + chunk]), 0), np.float32)
            ok = (S < thr) if strict else (S <= thr)
        if mask is not None:
            ok &= np.asarray(mask, bool)[None, :]
        for f in range(S.shape[0]):
            cand = np.nonzero(ok[f])[0]
            s = S[f, cand]
            order = np.lexsort((cand, s if metric == "euclidean" else -s))
            counts[a + f] = cand.size
            rows.append(cand[order].astype(np.int64))
            scores.append(s[order].astype(np.float32))
    return counts, rows, scores
