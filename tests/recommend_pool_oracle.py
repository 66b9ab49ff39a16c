"""fp64 oracle of retrieval from a pool with the classification-baseline blend (nrb_recommend_pool_blend).

Builds the fp64 score matrix that `recommend_oracle.check_lists` / `recommend_from_scores` take: NaN for rows outside
the pool, cos * alpha + base * (1 - alpha) for users with a history, base alone for users without one.
"""
from __future__ import annotations

import numpy as np


def pool_blend_scores(cos: np.ndarray, pool=None, base=None, alpha: float = 1.0, cold=None) -> np.ndarray:
    """fp64 [U, N] score matrix of nrb_recommend_pool_blend from the cosine matrix: NaN outside the pool; with a
    baseline, cos * alpha + base * (1 - alpha) for users with a history and base alone for `cold` users (bool [U])."""
    s = np.asarray(cos, dtype=np.float64).copy()
    if base is not None:
        b = np.asarray(base, dtype=np.float64)[None, :]
        with np.errstate(invalid="ignore"):
            s = s * np.float64(np.float32(alpha)) + b * np.float64(np.float32(1.0 - np.float32(alpha)))
        if cold is not None:
            s[np.asarray(cold, dtype=bool)] = b[0]
    if pool is not None:
        keep = np.zeros(s.shape[1], dtype=bool)
        keep[np.asarray(pool, dtype=np.int64)] = True
        s[:, ~keep] = np.nan
    return s


def naive_pool_blend(users: np.ndarray, table: np.ndarray, k: int, excl: list, pool=None, base=None,
                     alpha: float = 1.0, cold=None):
    """Per-user Python loop over the pool's rows: the pool / blend definition, spelled out."""
    U = users.shape[0]
    rows = np.full((U, k), -1, dtype=np.int32)
    out = np.full((U, k), np.nan)
    ids = range(table.shape[0]) if pool is None else sorted(set(int(r) for r in pool))
    a = float(np.float32(alpha))
    oma = float(np.float32(1.0 - np.float32(alpha)))
    for i in range(U):
        u = users[i].astype(np.float64)
        un = u / max(float(np.sqrt(np.dot(u, u))), 1e-8)
        cands = []
        for r in ids:
            if r in excl[i]:
                continue
            c = table[r].astype(np.float64)
            s = float(np.dot(un, c / max(float(np.sqrt(np.dot(c, c))), 1e-8)))
            if base is not None:
                s = float(base[r]) if (cold is not None and cold[i]) else s * a + float(base[r]) * oma
            s += 0.0
            if s != s:
                continue
            cands.append((-s, r))
        cands.sort()
        for j, (ns, r) in enumerate(cands[:k]):
            rows[i, j] = r
            out[i, j] = -ns
    return rows, out
