"""The vectorised references of tests/segment_oracle.py against the per-group definitions they restate (no GPU)."""
import numpy as np
import torch

from oracle import oracle
from tests import segment_oracle as so


def _groups(rng, n_groups, hi):
    counts = rng.integers(0, hi, size=n_groups).astype(np.int64)
    counts[:4] = [0, 1, 2, 700]
    return counts, so.csr(counts)


def test_dense_rank_segments_equals_rank_group_preds():
    rng = np.random.default_rng(0)
    counts, off = _groups(rng, 400, 40)
    for dtype in (np.float32, np.float64):
        scores = (rng.integers(-6, 7, size=int(off[-1])) / 4.0).astype(dtype)  # heavy ties
        scores[off[3]:off[3] + 50] = rng.standard_normal(50)
        scores[off[5]] = -0.0  # -0.0 == 0.0
        scores[off[5] + 1] = 0.0
        scores[off[9] + 1] = np.nan
        if dtype == np.float64:
            scores[off[11]:off[11] + 3] = [0.5, 0.5 + 1e-12, 0.5 - 1e-12]  # below fp32 resolution: distinct
        ranks, gap = so.dense_rank_segments(torch.from_numpy(scores), torch.from_numpy(off))
        gap = gap.numpy()
        want = np.nan_to_num(np.concatenate(oracle.rank_group_preds(scores, counts)), nan=0.0).astype(np.int32)
        assert np.array_equal(ranks.numpy(), want)
        for g in range(len(counts)):
            s = np.sort(scores[off[g]:off[g + 1]].astype(np.float64))
            if np.isnan(s).any():
                assert np.isnan(gap[g])
            else:
                assert gap[g] == (np.diff(s).min() if len(s) > 1 else np.inf)


def test_topk_order_segments_equals_stable_argsort():
    rng = np.random.default_rng(1)
    counts, off = _groups(rng, 300, 50)
    scores = (rng.integers(-6, 7, size=int(off[-1])) / 4.0).astype(np.float32)
    scores[[off[3] + 2, off[3] + 9, off[7]]] = np.nan
    scores[off[8]], scores[off[8] + 1] = 0.0, -0.0
    ks = (1, 5, 37)
    got = so.topk_order_segments(scores, counts, ks)
    for out, k in zip(got, ks):
        for g in range(len(counts)):
            s = scores[off[g]:off[g + 1]]
            order = np.argsort(-np.where(np.isnan(s), -np.inf, s), kind="stable")
            order = np.concatenate([order[~np.isnan(s[order])], order[np.isnan(s[order])]])
            want = np.full(k, -1, dtype=np.int32)
            want[:min(k, len(s))] = order[:k]
            assert np.array_equal(out[g], want), (g, k)


def _score_row_stable(y, ranks):
    """oracle.score_row with the stable tie order: np.argsort(..., kind="stable")[::-1]."""
    y = np.asarray(y, dtype=np.float64)
    ys = 1.0 / np.asarray(ranks, dtype=np.float64)
    order = np.argsort(ys, kind="stable")[::-1]
    ideal = np.argsort(y, kind="stable")[::-1]
    dcg = lambda o, k: np.sum((2 ** y[o[:k]] - 1) / np.log2(np.arange(len(o[:k])) + 2))
    mrr = np.sum(y[order] / (np.arange(len(y)) + 1)) / y.sum()
    return (oracle._auc_tie_aware(y, ys), mrr, dcg(order, 5) / dcg(ideal, 5), dcg(order, 10) / dcg(ideal, 10))


def test_mind_metrics_segments_equals_score_row():
    rng = np.random.default_rng(2)
    counts, off = _groups(rng, 300, 60)
    scores = rng.integers(0, 8, size=int(off[-1])).astype(np.float32)  # heavy ties
    ranks = np.concatenate([oracle.dense_rank_desc(scores[off[g]:off[g + 1]]) for g in range(len(counts))])
    labels = (rng.random(int(off[-1])) < 0.3).astype(np.int8)
    labels[off[1:-1][counts[1:] > 1]] = 1
    labels[off[1:-1][counts[1:] > 1] + 1] = 0
    labels[off[10]] = 2  # gains 2^y - 1
    labels[off[11]:off[12]] = 0  # single class
    labels[off[12]:off[13]] = 1
    ranks[off[13]:off[14]] = 0  # NaN group
    per = so.mind_metrics_segments(ranks, labels, counts)
    invalid = {11, 12, 13} | set(np.flatnonzero(counts < 2).tolist())  # one candidate or none: a single class
    for g in range(len(counts)):
        y, r = labels[off[g]:off[g + 1]], ranks[off[g]:off[g + 1]]
        if g in invalid:
            assert np.isnan(per[g]).all(), g
            continue
        np.testing.assert_allclose(per[g], _score_row_stable(y, r), atol=1e-12, rtol=0)
        # where tied candidates all carry the same label, the tie order cannot matter: the reference's own score_row
        if all(len(set(y[r == v])) == 1 for v in np.unique(r)):
            np.testing.assert_allclose(per[g], oracle.score_row(y, r), atol=1e-12, rtol=0)


def test_pool_score_fp64_equals_per_impression_oracle():
    g = torch.Generator().manual_seed(3)
    n_rows, d = 50, 16
    X, E, T = torch.randn(n_rows, d, generator=g), torch.randn(n_rows, d, generator=g).exp(), torch.randn(n_rows, d)
    base = torch.randn(n_rows, generator=g)
    rng = np.random.default_rng(3)
    hist_len = rng.integers(0, 9, size=40)
    cand_len = rng.integers(0, 7, size=40)
    hist_len[:2], cand_len[2] = 0, 0
    hist_idx = rng.integers(0, n_rows, size=int(hist_len.sum())).astype(np.int32)
    cand_idx = rng.integers(0, n_rows, size=int(cand_len.sum())).astype(np.int32)
    ho, co = so.csr(hist_len), so.csr(cand_len)
    t = torch.from_numpy
    for mode in (0, 1):
        for blend in (False, True):
            # small chunks: the chunking itself is under test
            user, scores = so.pool_score_fp64(mode, X, E, T, t(hist_idx), t(ho), t(cand_idx), t(co),
                                              base if blend else None, 0.7, max_elems=5 * d)
            for i in range(len(hist_len)):
                r = t(hist_idx[ho[i]:ho[i + 1]]).long()
                x = X.double()[r]
                if mode == 0:
                    e = E.double()[r]
                    u = (x * e).sum(0) / (e.sum(0) + 1e-10)
                else:
                    u = x.sum(0) / float(len(r))
                    u = u / u.norm().clamp_min(1e-12)
                assert torch.allclose(user[i], u, atol=1e-14, rtol=1e-12, equal_nan=True)
                want = oracle.cosine_scores(u[None], T, cand_idx[co[i]:co[i + 1]], cand_len[i:i + 1]).numpy()
                if blend:
                    b = base.double().numpy()[cand_idx[co[i]:co[i + 1]]]
                    want = 0.7 * want + 0.3 * b if hist_len[i] > 0 else b
                np.testing.assert_allclose(scores[co[i]:co[i + 1]].numpy(), want, atol=1e-14, rtol=0)
            if mode == 1:
                assert torch.isnan(user[:2]).all()
