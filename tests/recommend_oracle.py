"""fp64 oracle of whole-table retrieval (nrb_recommend) and the checks the GPU tests apply to its output.

score(u, r) = (u / max(|u|, 1e-8)) . c_r / max(|c_r|, 1e-8), order: score descending, equal scores by ascending row id
(-0.0 == 0.0), NaN never returned, excluded rows never returned, (-1, NaN) once a user's eligible rows run out.
"""
from __future__ import annotations

import numpy as np


def cosine_matrix(users: np.ndarray, table: np.ndarray) -> np.ndarray:
    """fp64 [U, N] cosine of every user against every row, both normalised by max(norm, 1e-8)."""
    u = np.asarray(users, dtype=np.float64)
    c = np.asarray(table, dtype=np.float64)
    un = u / np.maximum(np.linalg.norm(u, axis=1, keepdims=True), 1e-8)
    cn = c / np.maximum(np.linalg.norm(c, axis=1, keepdims=True), 1e-8)
    return un @ cn.T


def excluded_sets(excl_idx, excl_len, n_users: int) -> list:
    if excl_idx is None:
        return [set() for _ in range(n_users)]
    off = np.concatenate([[0], np.cumsum(np.asarray(excl_len, dtype=np.int64))])
    return [set(np.asarray(excl_idx)[off[i]:off[i + 1]].tolist()) for i in range(n_users)]


def recommend_from_scores(scores: np.ndarray, k: int, excl: list):
    """(rows int32 [U, k], scores float64 [U, k]) from a full fp64 score matrix."""
    U, N = scores.shape
    rows = np.full((U, k), -1, dtype=np.int32)
    out = np.full((U, k), np.nan)
    ids = np.arange(N)
    for i in range(U):
        s = scores[i] + 0.0  # -0.0 -> 0.0
        ok = ~np.isnan(s)
        if excl[i]:
            ok[np.fromiter(excl[i], dtype=np.int64)] = False
        cand = ids[ok]
        order = np.lexsort((cand, -s[cand]))[:k]
        rows[i, :len(order)] = cand[order]
        out[i, :len(order)] = s[cand[order]]
    return rows, out


def recommend(users: np.ndarray, table: np.ndarray, k: int, excl_idx=None, excl_len=None):
    """The fp64 reference result of nrb_recommend."""
    s = cosine_matrix(users, table)
    return recommend_from_scores(s, k, excluded_sets(excl_idx, excl_len, s.shape[0]))


def check_lists(rows: np.ndarray, scores: np.ndarray, ref_scores: np.ndarray, k: int, excl: list, bar: float):
    """The properties a returned [U, k] result must have against the fp64 score matrix of the same stored table:
    scores within `bar` of fp64, ordered, no duplicate / excluded rows, padding exactly when eligible rows run out,
    and every eligible row whose fp64 score beats the k-th returned score by more than 2 * bar present."""
    U, N = ref_scores.shape
    assert rows.shape == (U, k) and scores.shape == (U, k)
    for i in range(U):
        r, s = rows[i], scores[i]
        ref = ref_scores[i]
        elig = ~np.isnan(ref)
        if excl[i]:
            elig[np.fromiter(excl[i], dtype=np.int64)] = False
        n_elig = int(elig.sum())
        n_valid = int((r >= 0).sum())
        assert n_valid == min(k, n_elig), (i, n_valid, n_elig)
        assert np.all(r[:n_valid] >= 0) and np.all(r[n_valid:] == -1), i
        assert np.all(np.isnan(s[n_valid:])) and not np.any(np.isnan(s[:n_valid])), i
        got_r, got_s = r[:n_valid].astype(np.int64), s[:n_valid].astype(np.float64)
        assert len(set(got_r.tolist())) == n_valid, ("duplicate rows", i)
        assert not (set(got_r.tolist()) & excl[i]), ("excluded row returned", i)
        assert np.all(elig[got_r]), i
        np.testing.assert_allclose(got_s, ref[got_r], atol=bar, rtol=0, err_msg=f"user {i}")
        d = np.diff(got_s)
        assert np.all(d <= 0), ("not descending", i)
        tie = d == 0
        assert np.all(np.diff(got_r)[tie] > 0), ("ties not by ascending row", i)
        if n_valid == k and n_valid < n_elig:
            must = np.nonzero(elig & (ref > got_s[-1] + 2 * bar))[0]
            assert set(must.tolist()) <= set(got_r.tolist()), ("missing a clearly better row", i)


def naive_recommend(users: np.ndarray, table: np.ndarray, k: int, excl: list):
    """Per-user Python loop over every row: the definition, spelled out."""
    U = users.shape[0]
    rows = np.full((U, k), -1, dtype=np.int32)
    out = np.full((U, k), np.nan)
    for i in range(U):
        u = users[i].astype(np.float64)
        un = u / max(float(np.sqrt(np.dot(u, u))), 1e-8)
        cands = []
        for r in range(table.shape[0]):
            if r in excl[i]:
                continue
            c = table[r].astype(np.float64)
            s = float(np.dot(un, c / max(float(np.sqrt(np.dot(c, c))), 1e-8))) + 0.0
            if s != s:
                continue
            cands.append((-s, r))
        cands.sort()
        for j, (ns, r) in enumerate(cands[:k]):
            rows[i, j] = r
            out[i, j] = -ns
    return rows, out
