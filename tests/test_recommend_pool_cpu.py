"""Retrieval from a pool with the classification-baseline blend, without a GPU: the fp64 oracle against a per-user
loop, and the argument checks of the library, `ops`, the engine's host normalisation and the helper, all of which
raise before any device is touched."""
import numpy as np
import pytest
import torch

from tests import recommend_oracle as ro
from tests import recommend_pool_oracle as rpo


@pytest.mark.parametrize("seed,U,N,d,k,alpha", [(0, 6, 40, 8, 3, 0.7), (1, 7, 25, 4, 10, 1.0),
                                                (2, 4, 12, 6, 32, 0.0), (3, 6, 50, 16, 1, 0.35)])
def test_pool_blend_oracle_equals_naive_loop(seed, U, N, d, k, alpha):
    rng = np.random.default_rng(seed)
    table = rng.standard_normal((N, d))
    users = rng.standard_normal((U, d))
    users[-1, 0] = np.nan                          # a cold user with a NaN vector (mean-pool of an empty history)
    table[1] = table[0]                            # tied cosines
    base = rng.standard_normal(N).astype(np.float32)
    base[2] = np.nan                               # never returned
    base[5] = base[6]                              # ties for cold users: ascending row id
    pool = np.unique(rng.integers(0, N, size=max(1, N // 2)))
    cold = np.zeros(U, dtype=bool)
    cold[[0, U - 1]] = True
    h_len = rng.integers(0, 8, size=U)
    h_len[cold] = 0
    h_idx = rng.integers(0, N, size=int(h_len.sum()))
    excl = ro.excluded_sets(h_idx, h_len, U)
    for p, b in ((pool, base), (pool, None), (None, base)):
        ref = rpo.pool_blend_scores(ro.cosine_matrix(users, table), p, b, alpha, cold if b is not None else None)
        rows, scores = ro.recommend_from_scores(ref, k, excl)
        n_rows, n_scores = rpo.naive_pool_blend(users, table, k, excl, p, b, alpha, cold if b is not None else None)
        assert np.array_equal(rows, n_rows)
        np.testing.assert_allclose(scores, n_scores, rtol=0, atol=1e-12)
        ro.check_lists(rows, scores, ref, k, excl, 1e-6)
        if p is not None:
            assert set(rows[rows >= 0].tolist()) <= set(pool.tolist())
        if b is not None:
            assert 2 not in rows
            want = [r for r in np.lexsort((np.arange(N), -base.astype(np.float64)))
                    if not np.isnan(base[r]) and (p is None or r in set(pool.tolist()))][:k]
            assert rows[U - 1, :len(want)].tolist() == want  # cold: the baseline's top-k, NaN user or not


def test_library_rejects_bad_pool_arguments():
    from news_recommendation_project_v2_b200 import _lib
    lib = _lib.load()
    q = lib.nrb_recommend_pool_blend_workspace_bytes
    assert q(1, 256, 100, 4, 0, 10, -1) == lib.nrb_recommend_workspace_bytes(1, 256, 100, 4, 0, 10) > 0
    assert q(1, 256, 100, 4, 0, 10, 0) > 0 and q(1, 256, 100, 4, 0, 10, 100) > 0
    assert q(1, 256, 100, 4, 0, 10, 101) == 0 and b"at most n_rows" in lib.nrb_last_error()
    assert q(1, 256, 100, 4, 0, 33, 10) == 0 and b"k must be in [1, 32]" in lib.nrb_last_error()
    assert q(1, 96, 100, 4, 0, 10, 10) == 0 and b"multiple of 64" in lib.nrb_last_error()
    assert q(7, 256, 100, 4, 0, 10, 10) == 0 and b"precision" in lib.nrb_last_error()
    assert q(1, 256, 100, 0, 0, 10, 10) == 0
    args = lambda n_pool, pool: (1, 256, 100, 8, 256, 8, 256, 8, 256, 4, None, None, 0, 10, pool, n_pool, None, 1.0,
                                 None, 8, 8, 8, 8, 1 << 20, None)
    assert lib.nrb_recommend_pool_blend(*args(101, 8)) == -1 and b"at most n_rows" in lib.nrb_last_error()
    assert lib.nrb_recommend_pool_blend(*args(5, None)) == -1 and b"needs `pool`" in lib.nrb_last_error()


def test_ops_checks_pool_and_baseline_before_the_device():
    from news_recommendation_project_v2_b200 import _lib, ops
    table, users = torch.zeros(10, 64), torch.zeros(2, 64)
    bad = [
        (dict(pool=torch.zeros(3, dtype=torch.int64)), "pool must be a 1-D int32"),
        (dict(pool=torch.zeros(2, 2, dtype=torch.int32)), "pool must be a 1-D int32"),
        (dict(pool=np.arange(3, dtype=np.int32)), "pool must be a 1-D int32"),
        (dict(pool=torch.zeros(11, dtype=torch.int32)), "at most 10 entries"),
        (dict(cand_base=torch.zeros(10, dtype=torch.float64)), "cand_base must be a 1-D float32"),
        (dict(cand_base=torch.zeros(9)), "one entry per table row"),
        (dict(hist_off=torch.zeros(3, dtype=torch.int32)), "hist_off must be a 1-D int64"),
        (dict(hist_off=torch.zeros(4, dtype=torch.int64)), "U \\+ 1 entries"),
    ]
    for kw, msg in bad:
        with pytest.raises(_lib.NrbError, match=msg):
            ops.recommend(table, users, 5, **kw)


def test_host_pool_and_baseline_normalisation():
    from news_recommendation_project_v2_b200.engine import host_base, host_pool
    assert host_pool([7, 3, 3, 0, 9], 10).tolist() == [0, 3, 7, 9]
    assert host_pool([7, 3], 10).dtype == np.int32
    mask = np.zeros(10, dtype=bool)
    mask[[1, 4, 9]] = True
    assert host_pool(mask, 10).tolist() == [1, 4, 9]
    assert host_pool(np.array([], dtype=np.int64), 10).size == 0
    with pytest.raises(IndexError):
        host_pool([0, 10], 10)
    with pytest.raises(IndexError):
        host_pool([-1, 3], 10)
    with pytest.raises(ValueError, match="mask over the 10"):
        host_pool(np.ones(9, dtype=bool), 10)
    with pytest.raises(ValueError, match="integer row ids"):
        host_pool(np.array([0.5, 2.0]), 10)
    with pytest.raises(ValueError, match="integer row ids"):
        host_pool(np.zeros((2, 2), dtype=np.int32), 10)
    assert host_base(np.arange(10), 10).dtype == np.float32
    with pytest.raises(ValueError, match="one score per table row"):
        host_base(np.zeros(9), 10)


def test_helper_checks_before_the_device():
    from news_recommendation_project_v2_b200.data_model_helper import get_top_k_recommendations
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention
    model = FinalAttention(64, 64, precision="fp32")
    table = torch.zeros(10, 64)
    h_idx, h_len = np.array([1, 2], dtype=np.int32), np.array([2])
    with pytest.raises(ValueError, match="history_bool needs classification_score"):
        get_top_k_recommendations(h_idx, h_len, table, model, k=3, history_bool=np.array([True, False]))
    with pytest.raises(ValueError, match="one score per table row"):
        get_top_k_recommendations(h_idx, h_len, table, model, k=3, classification_score=np.zeros(9))
    with pytest.raises(IndexError):
        get_top_k_recommendations(h_idx, h_len, table, model, k=3, pool=np.array([3, 12]))
