"""GPU parity: Stage B/C kernels (gather, pooling, cosine, dense rank) vs the CPU oracle.

Everything goes through the C ABI (ops.* -> libnrb200.so).  Integer / index outputs must be
bit-exact; floating point within the tolerance written next to each check.
"""
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from news_recommendation_project_v2_b200 import synthetic as syn
from tests import segment_oracle as so

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from news_recommendation_project_v2_b200 import ops as _ops
    return _ops


def _csr(lengths):
    return torch.from_numpy(syn.csr_offsets(np.asarray(lengths))).cuda()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_dense_rank_bit_exact(ops, golden_dir):
    g = np.load(os.path.join(golden_dir, "small_cases.npz"))
    ranks = ops.dense_rank(torch.from_numpy(g["rank_scores"]).cuda(), _csr(g["rank_counts"])).cpu().numpy()
    want = np.nan_to_num(g["rank_out"], nan=0.0).astype(np.int32)  # NaN group -> 0 sentinel
    assert np.array_equal(ranks, want)
    # random groups with heavy ties, empty groups and one group above the shared-memory capacity (512)
    rng = np.random.default_rng(0)
    counts = np.concatenate([rng.integers(0, 70, size=300), [700, 513, 512, 0, 1]]).astype(np.int32)
    scores = rng.integers(-5, 6, size=int(counts.sum())).astype(np.float32) / 4.0
    got =ops.dense_rank(torch.from_numpy(scores).cuda(), _csr(counts)).cpu().numpy()
    want = np.concatenate([np.asarray(r) for r in oracle.rank_group_preds(scores, counts)] + [np.zeros(0)])
    assert np.array_equal(got, want.astype(np.int32))
    # continuous scores: ranks are a permutation 1..n per group
    scores = rng.standard_normal(int(counts.sum())).astype(np.float32)
    got = ops.dense_rank(torch.from_numpy(scores).cuda(), _csr(counts)).cpu().numpy()
    want = np.concatenate([np.asarray(r) for r in oracle.rank_group_preds(scores, counts)])
    assert np.array_equal(got, want.astype(np.int32))
    # every warp on >= 3 groups: fp32 scores run on SMs x 32 CTAs of 8 warps, float64 on SMs x 32 CTAs of 4 warps;
    # the reference ranks all groups at once (tests/segment_oracle.py, held to rank_group_preds on the CPU)
    W = _sms() * 32 * 8
    n_groups = 3 * W + 1001
    assert n_groups // W >= 3 and n_groups // (_sms() * 32 * 4) >= 3
    counts = rng.integers(0, 70, size=n_groups).astype(np.int64)
    counts[[5, W + 5, 2 * W + 6, 3 * W + 7]] = [700, 0, 513, 1000]  # global-memory path / empty, next to small groups
    off = syn.csr_offsets(counts)
    n = int(off[-1])
    for dt in (np.float32, np.float64):
        scores = (rng.integers(-8, 9, size=n) / 4.0).astype(dt)  # heavy ties
        scores[n // 2:] = rng.standard_normal(n - n // 2)
        if dt == np.float64:  # differences below fp32 resolution stay distinct
            scores[: n // 2] += rng.integers(0, 2, size=n // 2) * 2.0 ** -40
        scores[[off[W + 9] + 1, off[2 * W + 6] + 100]] = np.nan  # NaN groups rank 0 (one on the global path)
        sc = torch.from_numpy(scores).cuda()
        want, _ = so.dense_rank_segments(sc, torch.from_numpy(off).cuda())
        assert torch.equal(ops.dense_rank(sc, torch.from_numpy(off).cuda()), want)


def test_gather_collate_bit_exact(ops, golden_dir):
    g = np.load(os.path.join(golden_dir, "small_cases.npz"))
    t = torch.Generator().manual_seed(7)
    table = torch.randn(11, 8, generator=t)
    groups = [np.array([3, 1, 4], dtype=np.int32), np.array([10], dtype=np.int32),
              np.array([0, 0, 5, 9, 2], dtype=np.int32), np.array([7, 8], dtype=np.int32)]
    lens = [len(x) for x in groups]
    emb, mask = ops.gather_collate(table.cuda(), torch.from_numpy(np.concatenate(groups)).cuda(), _csr(lens), max(lens))
    assert np.array_equal(emb.cpu().numpy(), g["collate_emb"])  # exact copies / exact zeros
    assert np.array_equal(mask.cpu().numpy(), g["collate_mask"]) and mask.dtype == torch.int32
    # larger random case, both dtypes
    for dt in (torch.float32, torch.bfloat16):
        table = syn.make_table(500, 768).to(dt)
        imp = syn.make_impressions(40, 500, h_max=50, seed=3)
        want_e, want_m = oracle.final_attention_eval_collate(oracle.group_items(imp.hist_idx, imp.hist_len), table)
        emb, mask = ops.gather_collate(table.cuda(), torch.from_numpy(imp.hist_idx).cuda(), _csr(imp.hist_len),
                                       int(imp.hist_len.max()))
        assert torch.equal(emb.cpu(), want_e.to(dt)) and torch.equal(mask.cpu(), want_m)
    # every warp of the grid (SMs x 32 CTAs of 8 warps, one warp per (group, slot)) on >= 4 slots
    W = _sms() * 32 * 8
    max_len = 64
    n_groups = -(-4 * W // max_len) + 3
    assert n_groups * max_len >= 4 * W
    rng = np.random.default_rng(4)
    lens = rng.integers(0, max_len + 1, size=n_groups).astype(np.int64)
    lens[[1, n_groups // 2]] = [max_len, 0]
    idx = torch.from_numpy(rng.integers(0, 5000, size=int(lens.sum())).astype(np.int32)).cuda()
    valid = torch.arange(max_len, device="cuda")[None, :] < torch.from_numpy(lens).cuda()[:, None]
    for dt in (torch.float32, torch.bfloat16):
        big = syn.make_table(5000, 256, seed=8).to(dt).cuda()
        emb, mask = ops.gather_collate(big, idx, _csr(lens), max_len)
        want = torch.zeros(n_groups, max_len, 256, dtype=dt, device="cuda")
        want[valid] = big[idx.long()]
        assert torch.equal(emb, want) and torch.equal(mask, valid.to(torch.int32))
    with pytest.raises(IndexError):
        ops.gather_collate(table.cuda(), torch.tensor([1, 500], dtype=torch.int32).cuda(), _csr([2]), 2)


def _oracle_pool_score(X, E, T, imp, mode):
    """fp64 oracle of the fused kernel given the SAME (already rounded) tables."""
    X, E, T = X.double(), (E.double() if E is not None else None), T.double()
    h_off, c_off = syn.csr_offsets(imp.hist_len), syn.csr_offsets(imp.cand_len)
    users = []
    for i in range(imp.n):
        r = torch.from_numpy(imp.hist_idx[h_off[i]:h_off[i + 1]]).long()
        if mode == 0:
            u = (X[r] * E[r]).sum(0) / (E[r].sum(0) + 1e-10)
        else:
            u = X[r].sum(0) / float(len(r))
            u = u / u.norm().clamp_min(1e-12)
        users.append(u)
    users = torch.stack(users)
    scores = oracle.cosine_scores(users, T, imp.cand_idx, imp.cand_len, dtype=torch.float64)
    return users, scores.numpy()


# every (dtype, vectors per lane) instantiation: NV = dim * elemsize / 512 = 1..8
@pytest.mark.parametrize("dtype,dim", [(torch.float32, 768), (torch.bfloat16, 768), (torch.bfloat16, 1024),
                                       (torch.float32, 1024), (torch.bfloat16, 256), (torch.float32, 128)] +
                         [(torch.bfloat16, d) for d in (512, 1280, 1536, 1792, 2048)] +
                         [(torch.float32, d) for d in (256, 384, 512, 640, 896)])
@pytest.mark.parametrize("mode,blend", [(0, False), (1, False), (0, True)], ids=["0", "1", "0-blend"])
def test_score_rank_vs_oracle(ops, dtype, dim, mode, blend):
    n_rows, n_imp = 3000, 257
    g = torch.Generator().manual_seed(11)
    T = syn.make_table(n_rows, dim, seed=5).to(dtype)
    X = torch.randn(n_rows, dim, generator=g).to(dtype)
    E = torch.exp(0.5 * torch.randn(n_rows, dim, generator=g)).to(dtype) if mode == 0 else None
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand="large", seed=17)
    rng = np.random.default_rng(1)
    # candidate counts around the in-smem rank capacity (512) and above it
    imp.cand_len[3:7] = [600, 511, 512, 513]
    imp.cand_idx = rng.integers(0, n_rows, size=int(imp.cand_len.sum())).astype(np.int32)
    # history lengths at the edges of the kernel's load batches (HR rows in flight) and of its 32-row blocks
    nv = dim * T.element_size() // 512
    hr = max(1, 16 // (nv * (2 if mode == 0 else 1)))
    imp.hist_len[10:17] = [1, hr, hr + 1, 32, 33, 64, 65]
    if blend:
        imp.hist_len[20:22] = 0  # no history: the baseline alone
    imp.hist_idx = rng.integers(0, n_rows, size=int(imp.hist_len.sum())).astype(np.int32)
    base = torch.randn(n_rows, generator=g) if blend else None
    alpha = 0.7 if blend else 1.0
    n_c = int(imp.cand_len.sum())
    user, scores, ranks = ops.score_rank(
        mode, X.cuda(), None if E is None else E.cuda(), T.cuda(), torch.from_numpy(imp.hist_idx).cuda(),
        _csr(imp.hist_len), torch.from_numpy(imp.cand_idx).cuda(), _csr(imp.cand_len), n_c, want_user=True,
        cand_base=None if base is None else base.cuda(), blend_alpha=alpha)
    want_u, want_s = _oracle_pool_score(X, E, T, imp, mode)
    if blend:  # alpha * cos + (1 - alpha) * base; impressions without history get the base alone
        b = base.double().numpy()[imp.cand_idx]
        has_hist = np.repeat(imp.hist_len > 0, imp.cand_len)
        want_s = np.where(has_hist, alpha * want_s + (1 - alpha) * b, b)
    # fp32 accumulation of <= 50 rows / dot products of length d: 1e-5 abs on O(1) values
    np.testing.assert_allclose(user.cpu().numpy(), want_u.float().numpy(), atol=2e-5, rtol=2e-5)
    np.testing.assert_allclose(scores.cpu().numpy(), want_s, atol=5e-6, rtol=0)
    # dense ranks: bit-exact given the kernel's own score bits ...
    got_r = ranks.cpu().numpy()
    want_r = np.concatenate(oracle.rank_group_preds(scores.cpu().numpy(), imp.cand_len)).astype(np.int32)
    assert np.array_equal(got_r, want_r)
    # ... and equal to the fp64 oracle's ranks wherever adjacent fp64 scores are > 1e-5 apart
    oracle_r = np.concatenate(oracle.rank_group_preds(want_s, imp.cand_len)).astype(np.int32)
    off = syn.csr_offsets(imp.cand_len)
    bad = 0
    for i in range(imp.n):
        s = np.sort(want_s[off[i]:off[i + 1]])
        if len(s) > 1 and np.min(np.diff(s)) <= 1e-5:
            continue
        bad += int(not np.array_equal(got_r[off[i]:off[i + 1]], oracle_r[off[i]:off[i + 1]]))
    assert bad == 0


def test_score_rank_edge_cases(ops):
    dim, n_rows = 256, 64
    T = syn.make_table(n_rows, dim, seed=2)
    X = torch.randn(n_rows, dim)
    E = torch.exp(torch.randn(n_rows, dim))
    # empty history -> user 0 -> all scores 0 -> all rank 1; empty candidate list; duplicated candidates tie
    hist_len = np.array([0, 3, 2], dtype=np.int32)
    hist_idx = np.array([1, 2, 3, 4, 5], dtype=np.int32)
    cand_len = np.array([4, 0, 5], dtype=np.int32)
    cand_idx = np.array([9, 8, 7, 6, 10, 11, 10, 12, 11], dtype=np.int32)
    user, scores, ranks = ops.score_rank(0, X.cuda(), E.cuda(), T.cuda(), torch.from_numpy(hist_idx).cuda(),
                                         _csr(hist_len), torch.from_numpy(cand_idx).cuda(), _csr(cand_len), 9,
                                         want_user=True)
    s, r = scores.cpu().numpy(), ranks.cpu().numpy()
    assert np.all(s[:4] == 0) and np.array_equal(r[:4], [1, 1, 1, 1])
    assert torch.all(user[0] == 0)
    assert s[4] == s[6] and s[5] == s[8] and r[4] == r[6] and r[5] == r[8]
    assert sorted(set(r[4:].tolist())) == [1, 2, 3]
    # out-of-range ids raise like torch indexing
    bad = hist_idx.copy()
    bad[0] = n_rows
    with pytest.raises(IndexError):
        ops.score_rank(0, X.cuda(), E.cuda(), T.cuda(), torch.from_numpy(bad).cuda(), _csr(hist_len),
                       torch.from_numpy(cand_idx).cuda(), _csr(cand_len), 9)
    bad = cand_idx.copy()
    bad[-1] = -1
    with pytest.raises(IndexError):
        ops.score_rank(0, X.cuda(), E.cuda(), T.cuda(), torch.from_numpy(hist_idx).cuda(), _csr(hist_len),
                       torch.from_numpy(bad).cuda(), _csr(cand_len), 9)
    # mean-pool of an empty history is 0/0 = NaN (latent_attention.py:168) -> NaN scores -> rank sentinel 0
    user, scores, ranks = ops.score_rank(1, X.cuda(), None, T.cuda(), torch.from_numpy(hist_idx).cuda(),
                                         _csr(hist_len), torch.from_numpy(cand_idx).cuda(), _csr(cand_len), 9,
                                         want_user=True)
    assert torch.isnan(user[0]).all() and torch.isnan(scores[:4]).all() and np.all(ranks.cpu().numpy()[:4] == 0)
    assert not torch.isnan(scores[4:]).any()


def test_odd_widths_run_padded_and_oversized_rows_are_an_error(ops):
    """A width that is no 512-byte multiple (100 fp32 elements) runs on zero-padded tables and gives the cosine of
    the logical row; rows beyond the kernel's 4 KB are an error at the C ABI, not undefined behaviour."""
    from news_recommendation_project_v2_b200._lib import NrbError
    g = torch.Generator().manual_seed(3)
    T = torch.randn(8, 100, generator=g).cuda()
    one = lambda v: torch.tensor([v], dtype=torch.int32).cuda()
    user, scores, ranks = ops.score_rank(1, T, None, T, one(2), _csr([1]), one(5), _csr([1]), 1, want_user=True)
    want = torch.nn.functional.cosine_similarity(T[2].double(), T[5].double(), dim=0)
    assert user.shape == (1, 100) and abs(float(scores[0]) - float(want)) < 1e-6 and int(ranks[0]) == 1
    big = torch.randn(4, 1280).cuda()  # 5 KB rows
    with pytest.raises(NrbError):
        ops.score_rank(1, big, None, big, one(0), _csr([1]), one(1), _csr([1]), 1)


def test_topk_order_bit_exact(ops):
    """Top-k orderings against a stable numpy argsort: ties, groups shorter than k, > 512 candidates, NaN last."""
    rng = np.random.default_rng(9)
    counts = np.concatenate([rng.integers(0, 60, size=200), [700, 3, 0, 1]]).astype(np.int32)
    scores = (rng.integers(-6, 7, size=int(counts.sum())) / 4.0).astype(np.float32)  # heavy ties
    scores[5] = np.nan
    off = syn.csr_offsets(counts)
    for k in (1, 5, 10, 37):
        got = ops.topk_order(torch.from_numpy(scores).cuda(), _csr(counts), k).cpu().numpy()
        for g in range(len(counts)):
            s = scores[off[g]:off[g + 1]]
            key = np.where(np.isnan(s), -np.inf, s)  # NaN last, stable among equals
            order = np.argsort(-key, kind="stable")
            if np.isnan(s).any():  # NaNs after every number (incl. -inf-like), by position
                order = np.concatenate([order[~np.isnan(s[order])], order[np.isnan(s[order])]])
            want = np.full(k, -1, dtype=np.int32)
            want[:min(k, len(s))] = order[:k]
            assert np.array_equal(got[g], want), (g, k)
    # every warp of the grid (SMs x 32 CTAs of 8 warps) on >= 3 groups, most of them shorter than k = 37; the
    # reference orders all groups at once (tests/segment_oracle.py, held to the loop above on the CPU)
    W = _sms() * 32 * 8
    n_groups = 3 * W + 777
    assert n_groups // W >= 3
    counts = rng.integers(0, 60, size=n_groups).astype(np.int32)
    counts[[3, W + 3, 2 * W + 3]] = [700, 0, 2]
    off = syn.csr_offsets(counts)
    scores = (rng.integers(-6, 7, size=int(off[-1])) / 4.0).astype(np.float32)
    scores[[off[W + 4], off[2 * W + 5] + 1, off[3] + 600]] = np.nan
    ks = (1, 5, 10, 37)
    for k, want in zip(ks, so.topk_order_segments(scores, counts, ks)):
        got = ops.topk_order(torch.from_numpy(scores).cuda(), _csr(counts), k).cpu().numpy()
        assert np.array_equal(got, want), k


def test_rank_group_preds_float64_not_merged_below_fp32(ops):
    """scipy ranks float64 scores in float64 (data_utils.py:415): values closer than fp32 resolution stay distinct."""
    from news_recommendation_project_v2_b200.data_utils import rank_group_preds
    scores = np.array([0.5, 0.5 + 1e-12, 0.5 - 1e-12, 0.25, 1.0, 1.0 + 1e-13, 1.0, np.nan, 2.0], dtype=np.float64)
    counts = np.array([4, 3, 2], dtype=np.int32)
    got = rank_group_preds(scores, counts)
    want = oracle.rank_group_preds(scores, counts)
    for g, w in zip(got, want):
        assert np.array_equal(np.asarray(g, dtype=np.float64), np.asarray(w, dtype=np.float64), equal_nan=True)
    # the same bits rounded to fp32 DO tie (and the fp32 entry point says so)
    got32 = rank_group_preds(scores.astype(np.float32), counts)
    assert np.array_equal(np.asarray(got32[0]), np.array([1, 1, 1, 2], dtype=np.float32))
    rng = np.random.default_rng(5)
    counts = np.concatenate([rng.integers(1, 90, size=200), [600]]).astype(np.int32)
    scores = rng.standard_normal(int(counts.sum()))
    scores[::7] = scores[1::7][: len(scores[::7])]  # ties
    got = np.concatenate([np.asarray(r) for r in rank_group_preds(scores, counts)])
    want = np.concatenate([np.asarray(r) for r in oracle.rank_group_preds(scores, counts)])
    assert np.array_equal(got, want)


def test_cached_engine_never_returns_a_stale_table(ops):
    """The engine cache is valid only for the very same live table object (ADVICE r1)."""
    from news_recommendation_project_v2_b200 import engine
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention
    model = FinalAttention(256, 512, precision="fp32").eval()
    model.load_state_dict(syn.make_final_attention_state_dict(256, 512, seed=3))
    t1 = syn.make_table(300, 256, seed=1)
    e1 = engine.cached_engine(t1, model, precision="fp32")
    assert engine.cached_engine(t1, model, precision="fp32") is e1
    key = next(iter(engine._engine_cache))
    t2 = syn.make_table(300, 256, seed=2)
    # forge the situation the advisor described: same key, different (new) table object
    engine._engine_cache[key] = (e1, __import__("weakref").ref(t2), None)
    e2 = engine.cached_engine(t1, model, precision="fp32")
    assert e2 is not e1


def test_score_host_int16_ranks_equal_int32(ops):
    """Host path with int16 ranks on the wire == int32 ranks; a rank above 32767 raises instead of wrapping."""
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention
    model = FinalAttention(256, 512, precision="bf16").eval()
    model.load_state_dict(syn.make_final_attention_state_dict(256, 512, seed=3))
    table = syn.make_table(3000, 256, seed=1)
    imp = syn.make_impressions(5000, 3000, h_max=50, cand="large", seed=9)
    eng = ScoringEngine(table, model, precision="bf16")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    ho, co = t(syn.csr_offsets(imp.hist_len)), t(syn.csr_offsets(imp.cand_len))
    s32, r32 = eng.score_host(t(imp.hist_idx), ho, t(imp.cand_idx), co, n_chunks=7)
    r16 = torch.empty(r32.numel(), dtype=torch.int16).pin_memory()
    s16, r16 = eng.score_host(t(imp.hist_idx), ho, t(imp.cand_idx), co, ranks_out=r16, n_chunks=7)
    assert r16.dtype == torch.int16 and torch.equal(r16.to(torch.int32), r32) and torch.equal(s16, s32)
    flag = ops.new_err_flag(torch.device("cuda"))
    big = torch.arange(1, 40001, dtype=torch.int32, device="cuda")
    out = ops.narrow_ranks(big, torch.empty(40000, dtype=torch.int16, device="cuda"), flag)
    assert int(out[100]) == 101 and int(out[-1]) == 32767
    with pytest.raises(OverflowError):
        ops.raise_on_index_error(flag, "narrow")
    # past one pass of the grid-stride loop (SMs x 16 CTAs x 256 threads x 8 ranks), with a scalar tail (n % 8 = 3)
    n = 5_000_003
    assert n // 8 > _sms() * 16 * 256 and n % 8 != 0
    g = torch.Generator(device="cuda").manual_seed(6)
    ranks = torch.randint(1, 32768, (n,), dtype=torch.int32, device="cuda", generator=g)
    flag = ops.new_err_flag(torch.device("cuda"))
    out = ops.narrow_ranks(ranks, torch.empty(n, dtype=torch.int16, device="cuda"), flag)
    assert torch.equal(out.to(torch.int32), ranks) and int(flag.item()) == 0
    for at in (n - 11, n - 2):  # the second pass of the 8-wide loop, the scalar tail
        r = ranks.clone()
        r[at] = 40000
        flag = ops.new_err_flag(torch.device("cuda"))
        out = ops.narrow_ranks(r, torch.full((n,), -5, dtype=torch.int16, device="cuda"), flag)
        want = r.clamp_max(32767)
        assert torch.equal(out.to(torch.int32), want) and int(out[at]) == 32767
        with pytest.raises(OverflowError):
            ops.raise_on_index_error(flag, "narrow")
