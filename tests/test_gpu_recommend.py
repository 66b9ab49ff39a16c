"""GPU: whole-table retrieval (nrb_recommend, tensor-core GEMM with the fused top-k epilogue) against the fp64 oracle
on the same stored table.  Bars: 3e-3 for bf16, 1e-5 for fp32 / fp32x3 (split-bf16 operands)."""
import numpy as np
import pytest
import torch

from news_recommendation_project_v2_b200 import synthetic as syn
from tests import recommend_oracle as ro

pytestmark = pytest.mark.gpu

BAR = {torch.bfloat16: 3e-3, torch.float32: 1e-5}


@pytest.fixture(scope="module")
def ops():
    from news_recommendation_project_v2_b200 import ops as _ops
    return _ops


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _history(rng, U, N, h_max=40):
    h_len = rng.integers(0, h_max, size=U).astype(np.int32)
    h_idx = rng.integers(0, N, size=int(h_len.sum())).astype(np.int32)
    if len(h_idx) > 3:
        h_idx[1] = h_idx[0]  # duplicated ids
        h_idx[2] = h_idx[0]
    return h_idx, h_len


def _dev_csr(h_idx, h_len):
    off = torch.from_numpy(syn.csr_offsets(h_len)).cuda()
    return torch.from_numpy(np.ascontiguousarray(h_idx, dtype=np.int32)).cuda(), off


def _ref_scores(users, table):
    """fp64 cosine matrix on the device (the stored table, as the kernel reads it)."""
    u = users.double()
    c = table.double()
    un = u / u.norm(dim=1, keepdim=True).clamp_min(1e-8)
    cn = c / c.norm(dim=1, keepdim=True).clamp_min(1e-8)
    return (un @ cn.T).cpu().numpy()


def _run_and_check(ops, table, users, k, h_idx=None, h_len=None):
    excl_idx = excl_off = None
    if h_idx is not None:
        excl_idx, excl_off = _dev_csr(h_idx, h_len)
    rows, scores = ops.recommend(table, users, k, excl_idx=excl_idx, excl_off=excl_off)
    torch.cuda.synchronize()
    ref = _ref_scores(users, table)
    excl = ro.excluded_sets(h_idx, h_len, users.shape[0])
    ro.check_lists(rows.cpu().numpy(), scores.cpu().numpy(), ref, k, excl, BAR[table.dtype])
    return rows, scores


SHAPES = [  # (U, N, d, k, dtype)
    (1, 100, 256, 10, torch.bfloat16), (127, 1000, 256, 32, torch.bfloat16), (129, 4097, 256, 1, torch.bfloat16),
    (300, 1000, 256, 10, torch.bfloat16), (1, 4097, 384, 32, torch.bfloat16), (127, 100, 768, 10, torch.bfloat16),
    (129, 1000, 1024, 32, torch.bfloat16), (300, 4097, 384, 1, torch.bfloat16),
    (1, 1000, 256, 32, torch.float32), (127, 4097, 384, 10, torch.float32), (129, 100, 768, 1, torch.float32),
    (300, 1000, 1024, 32, torch.float32), (300, 100, 256, 32, torch.bfloat16),
]


@pytest.mark.parametrize("U,N,d,k,dtype", SHAPES)
def test_recommend_matches_fp64(ops, U, N, d, k, dtype):
    rng = np.random.default_rng(U * 7 + N + d + k)
    g = torch.Generator(device="cuda").manual_seed(U + N + d + k)
    table = torch.randn(N, d, device="cuda", generator=g).to(dtype)
    users = torch.randn(U, d, device="cuda", generator=g)
    h_idx, h_len = _history(rng, U, N)
    _run_and_check(ops, table, users, k, h_idx, h_len)
    _run_and_check(ops, table, users, k)  # nothing excluded


def test_many_segments_per_cta_pair(ops):
    """Every CTA pair works through >= 3 row-block segments and some row block is split over >= 2 pairs."""
    N, d, k = 1000, 256, 10
    n_units = _sms() // 2
    npr = -(-N // 256)
    m_tiles = 3 * n_units + 1
    U = m_tiles * 256 - 77
    T = m_tiles * npr
    starts = [c * T // n_units for c in range(n_units + 1)]
    blocks = [len(set(u // npr for u in range(starts[c], starts[c + 1]))) for c in range(n_units)]
    assert min(blocks) >= 3
    owners = [len({c for c in range(n_units) if starts[c] < (m + 1) * npr and starts[c + 1] > m * npr})
              for m in range(m_tiles)]
    assert max(owners) >= 2
    g = torch.Generator(device="cuda").manual_seed(5)
    table = torch.randn(N, d, device="cuda", generator=g).to(torch.bfloat16)
    users = torch.randn(U, d, device="cuda", generator=g)
    h_idx, h_len = _history(np.random.default_rng(5), U, N, h_max=12)
    _run_and_check(ops, table, users, k, h_idx, h_len)


@pytest.mark.parametrize("dtype,k", [(torch.bfloat16, 32), (torch.float32, 10)])
def test_mind_large_table(ops, dtype, k):
    N, d, U = 161013, 1024, 200
    table = syn.make_table(N, d, seed=11).cuda().to(dtype)
    g = torch.Generator(device="cuda").manual_seed(12)
    users = torch.randn(U, d, device="cuda", generator=g)
    h_idx, h_len = _history(np.random.default_rng(12), U, N, h_max=60)
    _run_and_check(ops, table, users, k, h_idx, h_len)


def test_ties_zero_and_nan_users_long_history(ops):
    N, d, k = 600, 256, 32
    g = torch.Generator(device="cuda").manual_seed(3)
    table = torch.randn(N, d, device="cuda", generator=g).to(torch.bfloat16)
    table[100:110] = table[7]  # duplicated rows: equal scores, ascending ids
    users = torch.randn(6, d, device="cuda", generator=g)
    users[1] = table[7].float()  # rows 7, 100..109 tie at the top
    users[2] = 0.0
    users[3, 5] = float("nan")
    rng = np.random.default_rng(3)
    lens = np.array([3, 2, 4, 1, 5000, 0], dtype=np.int32)  # a 5,000-id history (sorted in several passes)
    h_idx = rng.integers(0, N, size=int(lens.sum())).astype(np.int32)
    h_idx[3:5] = [105, 7]  # user 1 excludes two of the tied rows
    h_idx[10:5010] = rng.integers(0, 300, size=5000)  # user 4: (almost) every row below 300, many times over
    rows, scores = _run_and_check(ops, table, users, k, h_idx, lens)
    rows, scores = rows.cpu().numpy(), scores.cpu().numpy()
    assert rows[1, :9].tolist() == [100, 101, 102, 103, 104, 106, 107, 108, 109]
    zero_excl = set(h_idx[5:9].tolist())
    assert rows[2].tolist() == [r for r in range(N) if r not in zero_excl][:k] and np.all(scores[2] == 0)
    assert np.all(rows[3] == -1) and np.all(np.isnan(scores[3]))
    assert np.all(rows[4] >= 0)
    assert not set(rows[4].tolist()) & set(h_idx[10:5010].tolist())


def test_fewer_eligible_rows_than_k(ops):
    N, d = 20, 128
    table = torch.randn(N, d, device="cuda").to(torch.bfloat16)
    users = torch.randn(3, d, device="cuda")
    h_idx = np.arange(15, dtype=np.int32)
    lens = np.array([15, 0, 0], dtype=np.int32)
    rows, _ = _run_and_check(ops, table, users, 32, h_idx, lens)
    r = rows.cpu().numpy()
    assert (r[0] >= 0).sum() == 5 and (r[1] >= 0).sum() == 20


def test_chunks_and_repeats_are_bit_identical(ops):
    N, d, k = 4097, 512, 10
    g = torch.Generator(device="cuda").manual_seed(9)
    table = torch.randn(N, d, device="cuda", generator=g).to(torch.bfloat16)
    users = torch.randn(3000, d, device="cuda", generator=g)
    h_idx, h_len = _history(np.random.default_rng(9), 3000, N)
    off = syn.csr_offsets(h_len)
    ei, eo = _dev_csr(h_idx, h_len)
    r_all, s_all = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo)
    r_again, s_again = ops.recommend(table, users, k, excl_idx=ei, excl_off=eo)
    assert torch.equal(r_all, r_again) and torch.equal(s_all.view(torch.int32), s_again.view(torch.int32))
    parts = []
    for i0 in range(0, 3000, 1000):
        ci, co = _dev_csr(h_idx[off[i0]:off[i0 + 1000]], h_len[i0:i0 + 1000])
        parts.append(ops.recommend(table, users[i0:i0 + 1000].contiguous(), k, excl_idx=ci, excl_off=co))
    assert torch.equal(torch.cat([p[0] for p in parts]), r_all)
    assert torch.equal(torch.cat([p[1] for p in parts]).view(torch.int32), s_all.view(torch.int32))


def test_out_of_range_history_raises(ops):
    table = torch.randn(50, 64, device="cuda").to(torch.bfloat16)
    users = torch.randn(2, 64, device="cuda")
    ei, eo = _dev_csr(np.array([3, 50], dtype=np.int32), np.array([1, 1], dtype=np.int32))
    with pytest.raises(IndexError):
        ops.recommend(table, users, 5, excl_idx=ei, excl_off=eo)


def _final_model(dim, hidden, seed, precision):
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention
    m = FinalAttention(dim, hidden, precision=precision)
    m.load_state_dict(syn.make_final_attention_state_dict(dim, hidden, seed=seed), strict=True)
    return m.eval()


def _encoders(dim, precision):
    from news_recommendation_project_v2_b200.attention import NewAttention
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    fa = _final_model(dim, 256, 21, precision)
    lat = LatentAttentionModel(dim=dim, num_latents=32, heads=2, dim_head=64, precision=precision).eval()
    lat.load_state_dict(syn.make_latent_state_dict(dim, 32, heads=2, dim_head=64, seed=22))
    na = NewAttention(hidden_size=dim, num_hidden_layers=1, precision=precision).eval()
    return {"final": fa, "latent": lat, "new": na}


@pytest.mark.parametrize("precision", ["bf16", "fp32", "fp32x3"])
@pytest.mark.parametrize("dim", [256, 384])
@pytest.mark.parametrize("encoder", ["final", "latent", "new"])
def test_engine_encoders_agree_with_score_rank(encoder, dim, precision):
    """The engine's user vector against the stored table in fp64, and every returned (user, row) score against what
    score_rank gives that row as a candidate; empty histories: FinalAttention users score 0 everywhere (first k
    non-excluded rows), latent users pool to NaN (nothing)."""
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    n_rows, n_imp, k = 1500, 140, 10
    torch.manual_seed(dim)
    model = _encoders(dim, precision)[encoder]
    table = syn.make_table(n_rows, dim, seed=31)
    query = syn.make_table(n_rows, dim, seed=32) if encoder == "final" else None
    imp = syn.make_impressions(n_imp, n_rows, h_max=30, seed=33)
    hist_len = imp.hist_len.copy()
    hist_len[5] = 0
    hist_idx = np.delete(imp.hist_idx, np.arange(syn.csr_offsets(imp.hist_len)[5], syn.csr_offsets(imp.hist_len)[6]))
    eng = ScoringEngine(table, model, query, precision=precision)
    rows, scores = eng.recommend(hist_idx, hist_len, k)
    user = eng.user_vectors(hist_idx, hist_len)
    ref = _ref_scores(user, eng.cand)
    bar = BAR[eng.cand.dtype]
    excl = ro.excluded_sets(hist_idx, hist_len, n_imp)
    r_np, s_np = rows.cpu().numpy(), scores.cpu().numpy()
    ro.check_lists(r_np, s_np, ref, k, excl, bar)
    if encoder == "latent":
        assert np.all(r_np[5] == -1)
    elif encoder == "final":
        assert r_np[5].tolist() == list(range(k)) and np.all(s_np[5] == 0)
    # score_rank with the returned rows as candidates
    ok = r_np >= 0
    cand_len = ok.sum(axis=1).astype(np.int32)
    _, sr, _ = eng.score(hist_idx, hist_len, r_np[ok].astype(np.int32), cand_len, want_ranks=False)
    np.testing.assert_allclose(s_np[ok], sr.cpu().numpy(), atol=bar, rtol=0)
    # no exclusion: a superset of the eligible rows, scores never below the excluded run's
    rows2, scores2 = eng.recommend(hist_idx, hist_len, k, exclude_history=False)
    ro.check_lists(rows2.cpu().numpy(), scores2.cpu().numpy(), ref, k, ro.excluded_sets(None, None, n_imp), bar)


def test_helper_and_component_on_a_small_pipeline():
    from news_recommendation_project_v2_b200.components import TopKRecommendationComponent
    from news_recommendation_project_v2_b200.data_model_helper import get_top_k_recommendations
    from news_recommendation_project_v2_b200.engine import cached_engine
    dim, n_rows, n_imp, k = 256, 800, 50, 8
    model = _final_model(dim, 256, 41, "bf16")
    table = syn.make_table(n_rows, dim, seed=42)
    imp = syn.make_impressions(n_imp, n_rows, h_max=20, seed=43)
    out = get_top_k_recommendations(imp.hist_idx, imp.hist_len, table, model, k=k, precision="bf16")
    assert out["top_k_rows"].shape == (n_imp, k) and out["top_k_rows"].dtype == np.int32
    assert out["top_k_scores"].dtype == np.float32
    eng = cached_engine(table, model, None, precision="bf16")
    ref = _ref_scores(eng.user_vectors(imp.hist_idx, imp.hist_len), eng.cand)
    ro.check_lists(out["top_k_rows"], out["top_k_scores"], ref, k, ro.excluded_sets(imp.hist_idx, imp.hist_len, n_imp),
                   BAR[torch.bfloat16])
    news_list = [f"N{1000 + i}" for i in range(n_rows)]
    ctx = {"news_embeddings": table, "history_rev_ind_array": [imp.hist_idx], "history_len_list": imp.hist_len,
           "news_list": news_list}
    res = TopKRecommendationComponent(k=k, attention_model=model, precision="bf16").transform(ctx)
    assert np.array_equal(res["top_k_rows"], out["top_k_rows"])
    assert np.array_equal(res["top_k_scores"], out["top_k_scores"])
    assert res["top_k_news"][3, 0] == news_list[out["top_k_rows"][3, 0]]
    assert res["news_list"] is news_list
