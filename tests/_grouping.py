"""Reference answer of a grouping search (include/ragfin.h ragfin_search_grouped, DESIGN.md 7d) over exact scores, shared by
the CPU and GPU grouping suites.  Test infrastructure."""
import numpy as np


def grouped_topk(S: np.ndarray, codes: np.ndarray, n_groups: int, k: int, allow=None, id_base: int = 0):
    """Grouping search over exact scores S [nq, n] (or [n]): the k best groups, one hit per group.  The allowed rows
    are ordered by (score desc, row asc) and the first row of each code in [0, n_groups) is kept; rows with other codes
    are never returned.  Returns ids int64 [nq, k] and scores fp32 [nq, k], padded with (-1, -inf)."""
    S = np.atleast_2d(np.asarray(S, dtype=np.float32))
    codes = np.asarray(codes, dtype=np.int64)
    ok = (codes >= 0) & (codes < n_groups)
    if allow is not None:
        ok &= np.asarray(allow, dtype=bool)
    rows = np.flatnonzero(ok)
    ids = np.full((len(S), k), -1, dtype=np.int64)
    scores = np.full((len(S), k), -np.inf, dtype=np.float32)
    for qi, s in enumerate(S):
        order = rows[np.lexsort((rows, -s[rows].astype(np.float64)))]
        _, first = np.unique(codes[order], return_index=True)   # first occurrence of each code = the group's best row
        best = order[np.sort(first)][:k]
        ids[qi, :len(best)] = best + id_base
        scores[qi, :len(best)] = s[best]
    return ids, scores
