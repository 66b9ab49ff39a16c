"""Whole-table retrieval without a GPU: the fp64 oracle against its definition, argument checks of the library, and
the public calls refusing to run without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import recommend_oracle as ro


def _case(rng, U, N, d, ties):
    table = rng.standard_normal((N, d))
    users = rng.standard_normal((U, d))
    if ties:
        table[N // 2] = table[1]          # duplicated rows: equal scores, ascending ids
        table[N // 3] = 3.0 * table[1]    # same direction, other norm: equal cosine
        table[0] = 0.0                    # zero row: score 0 for everybody
        users[0] = 0.0                    # zero user: every score 0
        users[-1, 0] = np.nan             # NaN user: nothing eligible
    return users, table


@pytest.mark.parametrize("seed,U,N,d,k,ties", [(0, 5, 40, 8, 3, True), (1, 7, 25, 4, 10, True),
                                               (2, 4, 12, 6, 32, True), (3, 6, 50, 16, 1, False)])
def test_oracle_equals_naive_loop(seed, U, N, d, k, ties):
    rng = np.random.default_rng(seed)
    users, table = _case(rng, U, N, d, ties)
    h_len = rng.integers(0, 8, size=U)
    h_idx = rng.integers(0, N, size=int(h_len.sum()))
    if len(h_idx) > 2:
        h_idx[1] = h_idx[0]  # duplicated history id
    excl = ro.excluded_sets(h_idx, h_len, U)
    rows, scores = ro.recommend(users, table, k, h_idx, h_len)
    n_rows, n_scores = ro.naive_recommend(users, table, k, excl)
    assert np.array_equal(rows, n_rows)
    np.testing.assert_allclose(scores, n_scores, rtol=0, atol=1e-12)
    ro.check_lists(rows, scores, ro.cosine_matrix(users, table), k, excl, 1e-6)
    if ties:
        # the zero user gets the first k non-excluded rows in ascending order, the NaN user nothing
        want = [r for r in range(N) if r not in excl[0]][:k]
        assert rows[0, :len(want)].tolist() == want
        assert np.all(rows[-1] == -1) and np.all(np.isnan(scores[-1]))


def test_oracle_ties_and_negative_zero():
    table = np.array([[1.0, 0.0], [0.0, 1.0], [0.0, 1.0], [-1.0, 0.0], [0.0, -1.0]])
    users = np.array([[0.0, 1.0], [1.0, 0.0]])
    rows, scores = ro.recommend(users, table, 5)
    # user 0: rows 1, 2 (score 1), then rows 0 and 3 (+-0), then row 4
    assert rows[0].tolist() == [1, 2, 0, 3, 4]
    assert rows[1].tolist() == [0, 1, 2, 4, 3]
    rows, _ = ro.recommend(users, table, 4, np.array([2, 2, 0]), np.array([2, 1]))
    assert rows[0].tolist() == [1, 0, 3, 4] and rows[1].tolist() == [1, 2, 4, 3]


def test_library_rejects_bad_arguments_before_any_cuda_call():
    from news_recommendation_project_v2_b200 import _lib
    lib = _lib.load()
    args = lambda k, dim: (1, dim, 100, 8, dim, 8, dim, 8, dim, 4, None, None, 0, k, 8, 8, 8, 8, 1 << 20, None)
    for k in (0, 33):
        assert lib.nrb_recommend(*args(k, 256)) == -1
        msg = lib.nrb_last_error()
        assert b"k must be in [1, 32]" in msg and b"shared-memory" in msg
        assert lib.nrb_recommend_workspace_bytes(1, 256, 100, 4, 0, k) == 0
    assert lib.nrb_recommend(*args(10, 96)) == -1 and b"multiple of 64" in lib.nrb_last_error()
    assert lib.nrb_recommend_workspace_bytes(1, 96, 100, 4, 0, 10) == 0
    assert lib.nrb_recommend_workspace_bytes(7, 256, 100, 4, 0, 10) == 0 and b"precision" in lib.nrb_last_error()


def test_public_calls_raise_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    from news_recommendation_project_v2_b200 import _lib, ops
    from news_recommendation_project_v2_b200.components import TopKRecommendationComponent
    from news_recommendation_project_v2_b200.data_model_helper import get_top_k_recommendations
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention
    with pytest.raises(_lib.NrbError):
        ops.recommend(torch.zeros(10, 64), torch.zeros(2, 64), 5)
    with pytest.raises(_lib.NrbError, match=r"k must be in \[1, 32\]"):
        ops.recommend(torch.zeros(10, 64), torch.zeros(2, 64), 33)
    with pytest.raises(_lib.NrbError, match="multiple of 64"):
        ops.recommend(torch.zeros(10, 96), torch.zeros(2, 96), 5)
    model = FinalAttention(64, 64, precision="fp32")
    with pytest.raises(_lib.NrbError):
        get_top_k_recommendations(np.array([1, 2], dtype=np.int32), np.array([2]), torch.zeros(10, 64), model, k=3)
    comp = TopKRecommendationComponent(k=3, attention_model=model)
    ctx = {"news_embeddings": torch.zeros(10, 64), "history_rev_ind_array": [np.array([1, 2], dtype=np.int32)],
           "history_len_list": np.array([2]), "news_list": [f"N{i}" for i in range(10)]}
    with pytest.raises(_lib.NrbError):
        comp.transform(ctx)


def test_prototypes_cover_the_recommend_abi():
    from news_recommendation_project_v2_b200 import _lib
    assert "nrb_recommend" in _lib.PROTOTYPES and "nrb_recommend_workspace_bytes" in _lib.PROTOTYPES
    assert _lib.load().nrb_recommend_workspace_bytes.restype is C.c_size_t
