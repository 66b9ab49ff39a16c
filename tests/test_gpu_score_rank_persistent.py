"""score_rank_kernel with several impressions per warp, and with long histories / candidate lists, against fp64.

`nrb_score_rank` launches one-warp CTAs in a grid-stride loop, capped at SMs x 16 x NRB_SCORE_GRID_MULT (4) x 8 warps.
Past the cap a warp takes impressions w, w + W, w + 2W, ... and reuses its registers (the pooled user vector) and its
shared-memory rank staging for each of them.  These tests size every case from the SM count so that each warp does at
least three impressions, put special impressions (empty history, empty candidate list, 600 candidates, duplicated
ids, the first and last table rows) next to ordinary ones on the same warp, and check every impression against an fp64
reference that uses no nrb kernel (tests/segment_oracle.py).
"""
import numpy as np
import pytest
import torch

from news_recommendation_project_v2_b200 import synthetic as syn
from tests import segment_oracle as so

pytestmark = pytest.mark.gpu

N_ROWS = 3000
# the bars of test_score_rank_vs_oracle (fp32 accumulation of O(1) values).  Over all ~1.9 M scores of every case here,
# and over histories of up to 4,096 rows, one B200 (1,000 W power limit) measured at most 7.3e-7 on the user vectors
# and 2.5e-7 on the scores: 27x and 20x headroom, so the long lists keep the same bars
USER_TOL, SCORE_TOL = 2e-5, 5e-6


@pytest.fixture(scope="module")
def ops():
    from news_recommendation_project_v2_b200 import ops as _ops
    return _ops


def _score_warps(n_imp):
    """Warps of nrb_score_rank's grid, sized the way the launch sizes it (NRB_SCORE_WARPS 1, NRB_SCORE_GRID_MULT 4)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return min(n_imp, sms * (16 // 1) * 4 * 8)


SPECIAL_KINDS = ("empty_history", "empty_candidates", "cand600", "duplicates", "edge_rows")


@pytest.fixture(scope="module")
def layout():
    """~3.5 impressions per warp: histories of 1-8 rows, 2-12 candidates, and on a few warps a special impression
    first (w) or second (w + W), ordinary ones around it."""
    W = _score_warps(1 << 40)
    n_imp = 3 * W + W // 2
    rng = np.random.default_rng(2024)
    hist_len = rng.integers(1, 9, size=n_imp).astype(np.int64)
    cand_len = rng.integers(2, 13, size=n_imp).astype(np.int64)
    special = {}
    for k, kind in enumerate(SPECIAL_KINDS):
        for w in (k, 64 + k, W // 2 + k, W - 1 - k):
            special[w] = kind
        for w in (1000 + k, W - 100 - k):
            special[w + W] = kind
    content = {}
    for i, kind in special.items():
        h = rng.integers(0, N_ROWS, size=int(hist_len[i]))
        c = rng.integers(0, N_ROWS, size=int(cand_len[i]))
        if kind == "empty_history":
            h = h[:0]
        elif kind == "empty_candidates":
            c = c[:0]
        elif kind == "cand600":  # above the 512 scores staged in shared memory: the global-memory rank path
            c = rng.integers(0, N_ROWS, size=600)
        elif kind == "duplicates":
            h = np.array([7, 7, 7, 11, 7])
            c = np.array([5, 9, 5, 5, 9, 13, 5])
        else:
            h = np.array([0, N_ROWS - 1, 0])
            c = np.array([N_ROWS - 1, 0, 5, N_ROWS - 1, 0])
        hist_len[i], cand_len[i] = len(h), len(c)
        content[i] = (h, c)
    ho, co = so.csr(hist_len), so.csr(cand_len)
    hist_idx = rng.integers(0, N_ROWS, size=int(ho[-1])).astype(np.int32)
    cand_idx = rng.integers(0, N_ROWS, size=int(co[-1])).astype(np.int32)
    for i, (h, c) in content.items():
        hist_idx[ho[i]:ho[i + 1]] = h
        cand_idx[co[i]:co[i + 1]] = c
    kinds = {kind: np.array(sorted(i for i, v in special.items() if v == kind)) for kind in SPECIAL_KINDS}
    t = lambda a: torch.from_numpy(a).cuda()
    return dict(n_imp=n_imp, W=W, hist_len=hist_len, cand_len=cand_len, ho=ho, co=co, kinds=kinds,
                hist_idx=t(hist_idx), cand_idx=t(cand_idx), hist_off=t(ho), cand_off=t(co))


def _max_excess(got, want, rtol):
    """(max over elements of |got - want| - rtol * |want|, max |got - want|), both NaN where exactly one of the two
    is NaN; in row chunks of 16 M elements."""
    excess, err = -float("inf"), 0.0
    chunk = max(1, (1 << 24) // got.shape[1])
    for i in range(0, got.shape[0], chunk):
        g, w = got[i:i + chunk].double(), want[i:i + chunk]
        both = torch.isnan(g) & torch.isnan(w)
        if bool((torch.isnan(g) ^ torch.isnan(w)).any()):
            return float("nan"), float("nan")
        d = torch.where(both, 0.0, (g - w).abs())
        err = max(err, float(d.max()) if d.numel() else 0.0)
        x = d - rtol * torch.where(both, 0.0, w.abs())
        excess = max(excess, float(x.max()) if x.numel() else -float("inf"))
    return excess, err


def _check_against_fp64(mode, X, E, T, base, alpha, imp, user, scores, ranks):
    """Every impression: user vectors and scores within the bars, ranks bit-exact given the kernel's own score bits
    and equal to the fp64 ranks wherever adjacent fp64 scores are more than 1e-5 apart.  Returns the measured maxima
    and the impressions the fp64 rank check covered."""
    want_u, want_s = so.pool_score_fp64(mode, X.cuda(), None if E is None else E.cuda(), T.cuda(), imp["hist_idx"],
                                        imp["hist_off"], imp["cand_idx"], imp["cand_off"],
                                        None if base is None else base.cuda(), alpha)
    ex_u, err_u = _max_excess(user, want_u, rtol=USER_TOL)
    ex_s, err_s = _max_excess(scores[:, None], want_s[:, None], rtol=0.0)
    own_r, _ = so.dense_rank_segments(scores, imp["cand_off"])
    ref_r, gap = so.dense_rank_segments(want_s, imp["cand_off"])
    grp = torch.repeat_interleave(torch.arange(imp["n_imp"], device="cuda"), imp["cand_off"][1:] - imp["cand_off"][:-1])
    clear = gap > 1e-5  # includes groups of one candidate (gap inf)
    fp64_bad = int(((ranks != ref_r) & clear[grp]).sum())
    return dict(ex_u=ex_u, err_u=err_u, ex_s=ex_s, err_s=err_s, own_rank_bad=int((ranks != own_r).sum()),
                fp64_rank_bad=fp64_bad, fp64_rank_groups=int(clear.sum()))


def _assert_measured(m, user_tol=USER_TOL, score_tol=SCORE_TOL):
    assert m["ex_u"] <= user_tol, m
    assert m["ex_s"] <= score_tol, m
    assert m["own_rank_bad"] == 0 and m["fp64_rank_bad"] == 0, m


# the 16 (dtype, dim) pairs of test_score_rank_vs_oracle: every vectors-per-lane instantiation NV = 1..8 of both dtypes
DTYPE_DIMS = ([(torch.float32, 768), (torch.bfloat16, 768), (torch.bfloat16, 1024), (torch.float32, 1024),
               (torch.bfloat16, 256), (torch.float32, 128)] +
              [(torch.bfloat16, d) for d in (512, 1280, 1536, 1792, 2048)] +
              [(torch.float32, d) for d in (256, 384, 512, 640, 896)])
CASES = ([(dt, d, mode, False) for dt, d in DTYPE_DIMS for mode in (0, 1)] +
         [(torch.bfloat16, 1024, 0, True), (torch.float32, 640, 0, True)])


@pytest.mark.parametrize("dtype,dim,mode,blend", CASES,
                         ids=[f"{str(dt)[6:]}-{d}-{m}{'-blend' if b else ''}" for dt, d, m, b in CASES])
def test_score_rank_several_impressions_per_warp(ops, layout, dtype, dim, mode, blend):
    imp = layout
    n_imp, W = imp["n_imp"], imp["W"]
    assert _score_warps(n_imp) == W and n_imp // W >= 3  # every warp scores >= 3 impressions in one launch
    g = torch.Generator().manual_seed(dim + 10 * mode)
    T = syn.make_table(N_ROWS, dim, seed=dim).to(dtype)
    X = torch.randn(N_ROWS, dim, generator=g).to(dtype)
    E = torch.exp(0.5 * torch.randn(N_ROWS, dim, generator=g)).to(dtype) if mode == 0 else None
    base = torch.randn(N_ROWS, generator=g) if blend else None
    alpha = 0.7 if blend else 1.0
    n_c = int(imp["co"][-1])
    args = (X.cuda(), None if E is None else E.cuda(), T.cuda())
    kw = dict(cand_base=None if base is None else base.cuda(), blend_alpha=alpha)
    user, scores, ranks = ops.score_rank(mode, *args, imp["hist_idx"], imp["hist_off"], imp["cand_idx"],
                                         imp["cand_off"], n_c, want_user=True, **kw)
    m = _check_against_fp64(mode, X, E, T, base, alpha, imp, user, scores, ranks)
    print(f"\nscore/rank {dtype} d={dim} mode={mode} blend={blend}: {n_imp} impressions on {W} warps; max |user err| "
          f"{m['err_u']:.2e}, max |score err| {m['err_s']:.2e}; fp64 ranks checked on {m['fp64_rank_groups']} "
          f"impressions")

    # the special impressions, spelled out
    co = imp["co"]
    cpos = lambda i: slice(int(co[i]), int(co[i + 1]))
    for i in imp["kinds"]["empty_history"]:
        s, r = scores[cpos(i)], ranks[cpos(i)]
        if blend:  # the baseline alone, bit for bit
            assert torch.equal(s, base.cuda()[imp["cand_idx"][cpos(i)].long()])
        elif mode == 1:  # mean of nothing = 0 / 0 = NaN, and a NaN group ranks 0
            assert torch.isnan(user[i]).all() and torch.isnan(s).all() and bool((r == 0).all())
        else:
            assert bool((user[i] == 0).all()) and bool((s == 0).all()) and bool((r == 1).all())
    for i in imp["kinds"]["duplicates"]:
        s, r = scores[cpos(i)], ranks[cpos(i)]
        assert s[0] == s[2] == s[3] == s[6] and s[1] == s[4] and r[0] == r[2] == r[3] == r[6] and r[1] == r[4]
    for i in imp["kinds"]["edge_rows"]:
        s = scores[cpos(i)]
        assert s[0] == s[3] and s[1] == s[4]

    # the same arrays in launches of at most W impressions (one impression per warp): windows into the shared index
    # arrays, written into one output, bit-identical to the single launch
    s2 = torch.full_like(scores, float("nan"))
    r2 = torch.full_like(ranks, -7)
    users = []
    for i0 in range(0, n_imp, W):
        i1 = min(i0 + W, n_imp)
        u, _, _ = ops.score_rank(mode, *args, imp["hist_idx"], imp["hist_off"][i0:i1 + 1], imp["cand_idx"],
                                 imp["cand_off"][i0:i1 + 1], n_c, want_user=True, out_scores=s2, out_ranks=r2, **kw)
        users.append(u)
    assert torch.equal(s2.view(torch.int32), scores.view(torch.int32)) and torch.equal(r2, ranks)
    assert torch.equal(torch.cat(users).view(torch.int32), user.view(torch.int32))
    _assert_measured(m)


LONG_CASES = [(dt, mode) for dt in (torch.bfloat16, torch.float32) for mode in (0, 1)]


@pytest.mark.parametrize("dtype,mode", LONG_CASES, ids=[f"{str(dt)[6:]}-{m}" for dt, m in LONG_CASES])
def test_score_rank_long_histories_and_candidate_lists(ops, dtype, mode):
    """Histories of 200 (BASELINE configs[4]), 1,000 and 4,096 rows, candidate lists of 2,048 and 20,000 (the
    global-memory rank path, O(n^2) per warp) at d = 1024 (NV 4 bf16, 8 fp32), against the same fp64 reference and
    bars.  Measured on one B200: user vectors within 2.5e-7, scores within 1.8e-7 (fp32, 4,096-row histories).  The
    fp64 rank check only covers the short lists: 2,048 cosines of a few tenths always hold two closer than 1e-5."""
    dim, n_rows = 1024, 30000
    g = torch.Generator(device="cuda").manual_seed(77 + mode)
    T = torch.nn.functional.normalize(torch.randn(n_rows, dim, device="cuda", generator=g), dim=1).to(dtype)
    X = torch.randn(n_rows, dim, device="cuda", generator=g).to(dtype)
    E = torch.exp(0.5 * torch.randn(n_rows, dim, device="cuda", generator=g)).to(dtype) if mode == 0 else None
    hist_len = np.array([200, 1000, 4096, 200, 1000, 4096, 4096, 3, 200], dtype=np.int64)
    cand_len = np.array([2048, 2048, 2048, 20000, 20000, 20000, 30, 20000, 7], dtype=np.int64)
    rng = np.random.default_rng(5 + mode)
    ho, co = so.csr(hist_len), so.csr(cand_len)
    t = lambda a: torch.from_numpy(a).cuda()
    imp = dict(n_imp=len(hist_len), hist_idx=t(rng.integers(0, n_rows, size=int(ho[-1])).astype(np.int32)),
               cand_idx=t(rng.integers(0, n_rows, size=int(co[-1])).astype(np.int32)), hist_off=t(ho), cand_off=t(co))
    user, scores, ranks = ops.score_rank(mode, X, E, T, imp["hist_idx"], imp["hist_off"], imp["cand_idx"],
                                         imp["cand_off"], int(co[-1]), want_user=True)
    m = _check_against_fp64(mode, X, E, T, None, 1.0, imp, user, scores, ranks)
    print(f"\nlong lists {dtype} mode={mode}: max |user err| {m['err_u']:.2e}, max |score err| {m['err_s']:.2e}; fp64 "
          f"ranks checked on {m['fp64_rank_groups']} of {imp['n_imp']} impressions")
    _assert_measured(m)
