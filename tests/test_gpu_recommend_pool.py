"""GPU: retrieval from a pool of the table's rows with the classification-baseline blend (nrb_recommend_pool_blend:
gathered GEMM operand, NRB_EPI_TOPK_BLEND epilogue) against the fp64 oracle on the same stored table, bit-identity
with the plain call where the semantics coincide, and the engine / helper / component layers.  Bars: 3e-3 for bf16,
1e-5 for fp32 / fp32x3 (split-bf16 operands)."""
import numpy as np
import pytest
import torch

from news_recommendation_project_v2_b200 import synthetic as syn
from tests import recommend_oracle as ro
from tests import recommend_pool_oracle as rpo
from tests.test_gpu_recommend import BAR, SHAPES, _dev_csr, _encoders, _final_model, _history, _ref_scores, _sms

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from news_recommendation_project_v2_b200 import ops as _ops
    return _ops


def _pool(rng, N, n_pool):
    return np.sort(rng.choice(N, size=n_pool, replace=False)).astype(np.int32)


def _base(rng, N, scale=0.3):
    return (scale * rng.standard_normal(N)).astype(np.float32)


def _bits(t):
    return t.view(torch.int32)


def _run_and_check(ops, table, users, k, h_idx, h_len, pool=None, base=None, alpha=1.0, ref=None):
    """One call with history exclusion and the cold rule from the same CSR, checked against the fp64 oracle."""
    ei, eo = _dev_csr(h_idx, h_len)
    pool_d = None if pool is None else torch.from_numpy(pool).cuda()
    base_d = None if base is None else torch.from_numpy(base).cuda()
    rows, scores = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo, pool=pool_d, cand_base=base_d,
                                 blend_alpha=alpha, hist_off=eo)
    torch.cuda.synchronize()
    cos = _ref_scores(users, table) if ref is None else ref
    cold = np.asarray(h_len) == 0
    want = rpo.pool_blend_scores(cos, pool, base, alpha, cold if base is not None else None)
    excl = ro.excluded_sets(h_idx, h_len, users.shape[0])
    r, s = rows.cpu().numpy(), scores.cpu().numpy()
    ro.check_lists(r, s, want, k, excl, BAR[table.dtype])
    if pool is not None:
        assert np.isin(r[r >= 0], pool).all()
    return rows, scores


def _pool_sizes(N):
    return sorted({n for n in (1, 255, 256, 257, max(1, N // 8), N) if n <= N})


@pytest.mark.parametrize("U,N,d,k,dtype", SHAPES)
def test_pool_sizes_with_and_without_blend(ops, U, N, d, k, dtype):
    """Pools of 1, 255, 256, 257, N/8 and N rows on single CTAs (U <= 128) and CTA pairs, cosine and blended."""
    rng = np.random.default_rng(U * 11 + N + d + k)
    g = torch.Generator(device="cuda").manual_seed(U + N + d + k + 1)
    table = torch.randn(N, d, device="cuda", generator=g).to(dtype)
    users = torch.randn(U, d, device="cuda", generator=g)
    h_idx, h_len = _history(rng, U, N)
    h_len[::5] = 0  # cold users among warm ones
    h_idx = rng.integers(0, N, size=int(h_len.sum())).astype(np.int32)
    cos = _ref_scores(users, table)
    base = _base(rng, N)
    for n_pool in _pool_sizes(N):
        pool = _pool(rng, N, n_pool)
        _run_and_check(ops, table, users, k, h_idx, h_len, pool=pool, ref=cos)
        _run_and_check(ops, table, users, k, h_idx, h_len, pool=pool, base=base, alpha=0.6, ref=cos)
    _run_and_check(ops, table, users, k, h_idx, h_len, base=base, alpha=0.25, ref=cos)  # whole table, blended


def test_many_segments_per_cta_pair_on_a_pool(ops):
    """The pool's column count sets the schedule: every CTA pair works through >= 3 row-block segments and some row
    block is split over >= 2 pairs (the arithmetic of test_many_segments_per_cta_pair)."""
    N_table, n_pool, d, k = 1500, 1000, 256, 10
    n_units = _sms() // 2
    npr = -(-n_pool // 256)
    m_tiles = 3 * n_units + 1
    U = m_tiles * 256 - 77
    T = m_tiles * npr
    starts = [c * T // n_units for c in range(n_units + 1)]
    assert min(len(set(u // npr for u in range(starts[c], starts[c + 1]))) for c in range(n_units)) >= 3
    assert max(len({c for c in range(n_units) if starts[c] < (m + 1) * npr and starts[c + 1] > m * npr})
               for m in range(m_tiles)) >= 2
    rng = np.random.default_rng(6)
    g = torch.Generator(device="cuda").manual_seed(6)
    table = torch.randn(N_table, d, device="cuda", generator=g).to(torch.bfloat16)
    users = torch.randn(U, d, device="cuda", generator=g)
    h_idx, h_len = _history(rng, U, N_table, h_max=12)
    pool = _pool(rng, N_table, n_pool)
    cos = _ref_scores(users, table)
    _run_and_check(ops, table, users, k, h_idx, h_len, pool=pool, ref=cos)
    _run_and_check(ops, table, users, k, h_idx, h_len, pool=pool, base=_base(rng, N_table), alpha=0.5, ref=cos)


@pytest.mark.parametrize("U,dtype", [(100, torch.bfloat16), (300, torch.bfloat16), (200, torch.float32)])
def test_whole_table_pool_and_unit_alpha_are_bit_identical_to_the_plain_call(ops, U, dtype):
    N, d, k = 3000, 256, 32
    rng = np.random.default_rng(U)
    g = torch.Generator(device="cuda").manual_seed(U)
    table = torch.randn(N, d, device="cuda", generator=g).to(dtype)
    users = torch.randn(U, d, device="cuda", generator=g)
    h_idx, h_len = _history(rng, U, N)
    h_len = np.maximum(h_len, 1)  # nobody cold
    h_idx = rng.integers(0, N, size=int(h_len.sum())).astype(np.int32)
    ei, eo = _dev_csr(h_idx, h_len)
    r0, s0 = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo)
    everything = torch.arange(N, dtype=torch.int32, device="cuda")
    base = torch.from_numpy(_base(rng, N)).cuda()
    for kw in (dict(pool=everything), dict(cand_base=base, blend_alpha=1.0, hist_off=eo),
               dict(pool=everything, cand_base=base, blend_alpha=1.0, hist_off=eo)):
        r1, s1 = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo, **kw)
        assert torch.equal(r1, r0) and torch.equal(_bits(s1), _bits(s0)), kw.keys()
    # a pool with alpha = 1 is the same as the pool without a baseline
    pool = torch.from_numpy(_pool(rng, N, 700)).cuda()
    r2, s2 = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo, pool=pool)
    r3, s3 = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo, pool=pool, cand_base=base, blend_alpha=1.0,
                           hist_off=eo)
    assert torch.equal(r2, r3) and torch.equal(_bits(s2), _bits(s3))


@pytest.mark.parametrize("ends_in_pool", [True, False])
def test_histories_with_awkward_ids(ops, ends_in_pool):
    """Excluded ids inside and outside the pool, duplicated, and the first and last table rows."""
    N, d, k, U = 2000, 256, 32, 150
    rng = np.random.default_rng(17 + ends_in_pool)
    g = torch.Generator(device="cuda").manual_seed(17)
    table = torch.randn(N, d, device="cuda", generator=g).to(torch.bfloat16)
    users = torch.randn(U, d, device="cuda", generator=g)
    pool = _pool(rng, N, 300)
    pool = np.union1d(pool, [0, N - 1]) if ends_in_pool else np.setdiff1d(pool, [0, N - 1])
    pool = pool.astype(np.int32)
    h_len = rng.integers(1, 60, size=U).astype(np.int32)
    parts = []
    for i in range(U):
        inside = rng.choice(pool, size=h_len[i] // 2)
        outside = rng.integers(0, N, size=h_len[i] - h_len[i] // 2)
        ids = np.concatenate([inside, outside]).astype(np.int32)
        ids[0] = [0, N - 1, pool[0], pool[-1]][i % 4]
        if len(ids) > 2:
            ids[1] = ids[0]  # duplicated
        parts.append(rng.permutation(ids))
    # user 0: excludes every pool row -> all padding; user 1: every pool row but two or three
    parts[0] = np.concatenate([pool, pool[:5]]).astype(np.int32)
    parts[1] = np.concatenate([pool[3:], [0, N - 1]]).astype(np.int32)
    h_len = np.array([len(p) for p in parts], dtype=np.int32)
    h_idx = np.concatenate(parts).astype(np.int32)
    rows, _ = _run_and_check(ops, table, users, k, h_idx, h_len, pool=pool)
    r = rows.cpu().numpy()
    assert np.all(r[0] == -1)
    assert sorted(r[1][r[1] >= 0].tolist()) == sorted(set(pool.tolist()) - set(parts[1].tolist()))
    _run_and_check(ops, table, users, k, h_idx, h_len, pool=pool, base=_base(rng, N), alpha=0.3)


@pytest.mark.parametrize("precision", ["bf16", "fp32", "fp32x3"])
@pytest.mark.parametrize("encoder", ["final", "latent"])
def test_cold_users_among_warm_users_on_the_engine(encoder, precision):
    """Users without a history get the baseline's top-k of the pool, whatever their user vector (FinalAttention: the
    zero vector, latent mean-pool: NaN); users with one get the blend, and each returned score is what score_rank
    gives that row as a candidate with the same baseline."""
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    dim, n_rows, n_imp, k, alpha = 256, 1500, 140, 10, 0.65
    torch.manual_seed(7)
    model = _encoders(dim, precision)[encoder]
    table = syn.make_table(n_rows, dim, seed=51)
    imp = syn.make_impressions(n_imp, n_rows, h_max=30, seed=52)
    off = syn.csr_offsets(imp.hist_len)
    cold_ids = [0, 5, 77, n_imp - 1]
    keep = np.ones(len(imp.hist_idx), dtype=bool)
    for i in cold_ids:
        keep[off[i]:off[i + 1]] = False
    hist_idx, hist_len = imp.hist_idx[keep], imp.hist_len.copy()
    hist_len[cold_ids] = 0
    rng = np.random.default_rng(53)
    base = _base(rng, n_rows)
    base[rng.choice(n_rows, size=20, replace=False)] = np.nan  # rows never returned
    pool = rng.choice(n_rows, size=900)  # host ids with duplicates, any order
    eng = ScoringEngine(table, model, None, precision=precision)
    rows, scores = eng.recommend(hist_idx, hist_len, k, pool=pool, cand_base=base, blend_alpha=alpha)
    r_np, s_np = rows.cpu().numpy(), scores.cpu().numpy()
    user = eng.user_vectors(hist_idx, hist_len)
    cold = hist_len == 0
    want = rpo.pool_blend_scores(_ref_scores(user, eng.cand), np.unique(pool), base, alpha, cold)
    bar = BAR[eng.cand.dtype]
    ro.check_lists(r_np, s_np, want, k, ro.excluded_sets(hist_idx, hist_len, n_imp), bar)
    in_pool = set(pool.tolist())
    by_base = [r for r in np.lexsort((np.arange(n_rows), -base.astype(np.float64)))
               if not np.isnan(base[r]) and r in in_pool][:k]
    for i in cold_ids:
        assert r_np[i].tolist() == by_base and np.array_equal(s_np[i], base[by_base])
    ok = r_np >= 0
    _, sr, _ = eng.score(hist_idx, hist_len, r_np[ok].astype(np.int32), ok.sum(axis=1).astype(np.int32),
                         want_ranks=False, cand_base=base, blend_alpha=alpha)
    np.testing.assert_allclose(s_np[ok], sr.cpu().numpy(), atol=bar, rtol=0)
    # no exclusion: the cold rule still holds
    rows2, scores2 = eng.recommend(hist_idx, hist_len, k, exclude_history=False, pool=pool, cand_base=base,
                                   blend_alpha=alpha)
    ro.check_lists(rows2.cpu().numpy(), scores2.cpu().numpy(), want, k, ro.excluded_sets(None, None, n_imp), bar)
    assert rows2.cpu().numpy()[cold_ids[1]].tolist() == by_base


def test_bad_pools_and_nan_baseline(ops):
    N, d, k = 600, 128, 10
    g = torch.Generator(device="cuda").manual_seed(23)
    table = torch.randn(N, d, device="cuda", generator=g).to(torch.bfloat16)
    users = torch.randn(3, d, device="cuda", generator=g)
    for bad in ([3, 600], [-1, 4], [5, 4, 9], [2, 2, 3]):  # out of range, negative, descending, repeated
        with pytest.raises(IndexError):
            ops.recommend(table, users, k, pool=torch.tensor(bad, dtype=torch.int32, device="cuda"))
    ei, eo = _dev_csr(np.array([1, 600], dtype=np.int32), np.array([1, 1, 0], dtype=np.int32))
    with pytest.raises(IndexError):  # an excluded id outside the pool is still range-checked
        ops.recommend(table, users, k, excl_idx=ei, excl_off=eo, pool=torch.tensor([1, 2], dtype=torch.int32,
                                                                                    device="cuda"))
    # empty pool: all padding
    rows, scores = ops.recommend(table, users, k, pool=torch.zeros(0, dtype=torch.int32, device="cuda"))
    assert torch.all(rows == -1) and torch.all(torch.isnan(scores))
    # a NaN baseline row is never returned, not even to a user whose best row it would be
    base = torch.zeros(N, device="cuda")
    users[0] = table[42].float()
    base[42] = float("nan")
    off = torch.tensor([0, 0, 0, 0], dtype=torch.int64, device="cuda")  # everybody cold for the second call
    for hist_off in (None, off):
        rows, scores = ops.recommend(table, users, k, cand_base=base, blend_alpha=0.5, hist_off=hist_off)
        assert not (rows == 42).any() and not torch.isnan(scores).any()


def test_chunks_and_repeats_are_bit_identical(ops):
    N, d, k, U = 4097, 512, 10, 3000
    rng = np.random.default_rng(29)
    g = torch.Generator(device="cuda").manual_seed(29)
    table = torch.randn(N, d, device="cuda", generator=g).to(torch.bfloat16)
    users = torch.randn(U, d, device="cuda", generator=g)
    h_idx, h_len = _history(rng, U, N)
    off = syn.csr_offsets(h_len)
    pool = torch.from_numpy(_pool(rng, N, 1300)).cuda()
    base = torch.from_numpy(_base(rng, N)).cuda()
    ei, eo = _dev_csr(h_idx, h_len)
    kw = dict(pool=pool, cand_base=base, blend_alpha=0.4)
    r_all, s_all = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo, hist_off=eo, **kw)
    r_again, s_again = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo, hist_off=eo, **kw)
    assert torch.equal(r_all, r_again) and torch.equal(_bits(s_all), _bits(s_again))
    parts = []
    for i0 in range(0, U, 1000):
        ci, co = _dev_csr(h_idx[off[i0]:off[i0 + 1000]], h_len[i0:i0 + 1000])
        parts.append(ops.recommend(table, users[i0:i0 + 1000].contiguous(), k, excl_idx=ci, excl_off=co,
                                   hist_off=co, **kw))
    assert torch.equal(torch.cat([p[0] for p in parts]), r_all)
    assert torch.equal(_bits(torch.cat([p[1] for p in parts])), _bits(s_all))


def test_helper_and_component_with_pool_and_baseline():
    """get_top_k_recommendations and TopKRecommendationComponent end to end on a small MIND-shaped context: one list
    per behaviour row, users without a history on the baseline, the impressions' news as the pool; every retrieved
    score is the one get_final_score gives that news as a candidate."""
    from news_recommendation_project_v2_b200.components import TopKRecommendationComponent
    from news_recommendation_project_v2_b200.data_model_helper import (get_classification_preds, get_final_score,
                                                                       get_top_k_recommendations)
    from news_recommendation_project_v2_b200.modeling_utils import ClassificationHead, WeightedSumModel
    dim, n_rows, n_imp, k = 256, 800, 60, 8
    torch.manual_seed(61)
    model = _final_model(dim, 256, 61, "bf16")
    head = ClassificationHead(dim, dim, 1, precision="bf16").eval()
    wsum = WeightedSumModel()
    with torch.no_grad():
        wsum.alpha.fill_(0.4)
    table = syn.make_table(n_rows, dim, seed=62)
    imp = syn.make_impressions(n_imp, n_rows, h_max=20, seed=63)
    hb = np.ones(n_imp, dtype=bool)
    hb[[2, 9, 30]] = False
    off = syn.csr_offsets(imp.hist_len)
    hist_idx = np.concatenate([imp.hist_idx[off[i]:off[i + 1]] for i in np.flatnonzero(hb)]).astype(np.int32)
    hist_len = imp.hist_len[hb]  # history_* describe the rows with a history only
    cls = get_classification_preds(table, head)
    pool = np.unique(imp.cand_idx)
    out = get_top_k_recommendations(hist_idx, hist_len, table, model, k=k, precision="bf16", pool=pool,
                                    classification_score=cls, weight_model=wsum, history_bool=hb)
    rows, scores = out["top_k_rows"], out["top_k_scores"]
    assert rows.shape == (n_imp, k) and rows.dtype == np.int32 and scores.dtype == np.float32
    assert np.isin(rows[rows >= 0], pool).all()
    in_pool = set(pool.tolist())
    by_base = [r for r in np.lexsort((np.arange(n_rows), -cls.astype(np.float64))) if r in in_pool][:k]
    for i in np.flatnonzero(~hb):
        assert rows[i].tolist() == by_base
    # get_final_score with each user's retrieved news as the candidates of one impression
    ok = rows >= 0
    fs = get_final_score(hist_idx, hist_len, rows[ok].astype(np.int32), ok.sum(axis=1).astype(np.int32), table, cls,
                         hb, model, wsum, precision="bf16")
    np.testing.assert_allclose(scores[ok], fs["scores"], atol=BAR[torch.bfloat16], rtol=0)
    news_list = [f"N{1000 + i}" for i in range(n_rows)]
    ctx = {"news_embeddings": table, "history_rev_ind_array": [hist_idx], "history_len_list": hist_len,
           "news_list": news_list, "history_bool": hb, "impression_rev_ind_array": [imp.cand_idx]}
    comp = TopKRecommendationComponent(k=k, attention_model=model, precision="bf16", classification_model=head,
                                       weight_model=wsum, restrict_to_impressions=True)
    res = comp.transform(ctx)
    assert np.array_equal(res["top_k_rows"], rows) and np.array_equal(res["top_k_scores"], scores)
    assert res["top_k_news"][2, 0] == news_list[by_base[0]]
    # without the new arguments the component is the whole-table cosine of before
    plain = TopKRecommendationComponent(k=k, attention_model=model, precision="bf16").transform(ctx)
    want = get_top_k_recommendations(hist_idx, hist_len, table, model, k=k, precision="bf16")
    assert plain["top_k_rows"].shape == (len(hist_len), k)
    assert np.array_equal(plain["top_k_rows"], want["top_k_rows"])
    with pytest.raises(ValueError, match="history_bool needs classification_score"):
        get_top_k_recommendations(hist_idx, hist_len, table, model, k=k, history_bool=hb)
