"""Pin oracle/oracle.py against outputs of the reference itself (tests/golden,
minted by oracle/make_golden.py) -- CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from oracle.make_golden import sd_digest
from news_recommendation_project_v2_b200 import synthetic as syn


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"), allow_pickle=False)


@pytest.mark.parametrize("name", ["latent_cfg1_d768_L512", "latent_default_d1024_L64", "latent_cfg5_d1024_L1024"])
def test_latent_pool_matches_reference(golden_dir, name):
    g = _load(golden_dir, name)
    dim, L, B, S, seed = (int(g[k]) for k in ("dim", "L", "B", "S", "seed"))
    sd = syn.make_latent_state_dict(dim, L, seed=seed)
    assert sd_digest(sd) == str(g["sd_sha256"]), "weight generator drifted from the golden run"
    assert sorted(sd.keys()) == list(g["keys"])
    x, mask = syn.make_token_batch(B, S, dim, seed=seed + 1)
    pooled = oracle.latent_pool(sd, x, mask, dtype=torch.float64).float().numpy()
    # reference ran in fp32; oracle in fp64: tolerance = fp32 accumulation noise
    np.testing.assert_allclose(pooled, g["pooled"], atol=2e-6, rtol=0)
    un = oracle.latent_pool(sd, x[:1], None, dtype=torch.float64)[0].float().numpy()
    np.testing.assert_allclose(un, g["unpooled0"], atol=2e-4, rtol=1e-5)
    # fp32 oracle as well (the dtype the reference computes in)
    pooled32 = oracle.latent_pool(sd, x, mask, dtype=torch.float32).numpy()
    np.testing.assert_allclose(pooled32, g["pooled"], atol=2e-6, rtol=0)


def test_latent_pool_mask_semantics():
    sd = syn.make_latent_state_dict(64, 16, heads=2, dim_head=32, seed=5)
    x, mask = syn.make_token_batch(3, 6, 64, seed=6, min_len=2)
    base = oracle.latent_pool(sd, x, mask, heads=2, dim_head=32)
    x2 = x.clone()
    x2[mask == 0] = 123.0  # padded tokens never influence the output (SURVEY 3.2)
    assert torch.equal(base, oracle.latent_pool(sd, x2, mask, heads=2, dim_head=32))
    m0 = mask.clone()
    m0[1] = 0
    out = oracle.latent_pool(sd, x, m0, heads=2, dim_head=32)
    assert torch.isnan(out[1]).all() and not torch.isnan(out[0]).any()


@pytest.mark.parametrize("name", ["final_small_d768", "final_large_d1024"])
def test_final_attention_score_rank_matches_reference(golden_dir, name):
    g = _load(golden_dir, name)
    dim, hidden, n_rows, n_imp, seed = (int(g[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    sd = syn.make_final_attention_state_dict(dim, hidden, seed=seed)
    assert sd_digest(sd) == str(g["sd_sha256"])
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand=str(g["cand"]), seed=seed + 3)
    out = oracle.final_second_attention_score(sd, table, imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len,
                                              dtype=torch.float64)
    np.testing.assert_allclose(out["user"].float().numpy(), g["user"], atol=3e-6, rtol=1e-5)
    np.testing.assert_allclose(out["scores"], g["scores"], atol=2e-6, rtol=0)
    ranks = np.concatenate(out["grouped_scores"])
    ref_ranks = g["ranks"]
    # fp64 oracle vs fp32 reference: ranks may differ only where adjacent scores are within noise
    bad = np.flatnonzero(ranks != ref_ranks)
    assert len(bad) <= 2, f"{len(bad)} rank mismatches"
    # ranks from the reference's own score bits must be bit-exact
    ranks_from_ref_scores = np.concatenate(oracle.rank_group_preds(g["scores"], imp.cand_len))
    assert np.array_equal(ranks_from_ref_scores, ref_ranks)
    # metrics from the reference's ranks
    grouped = oracle.group_items(ref_ranks, imp.cand_len)
    m = np.array([oracle.score_row(imp.labels[i], grouped[i]) for i in range(n_imp)])
    np.testing.assert_allclose(m, g["metrics"], atol=1e-12, rtol=0)


def test_final_attention_medium_fixture_matches_reference(golden_dir):
    """1,024 impressions / 39 k candidates through the unmodified reference: oracle scores within 2e-6, dense ranks
    from the reference's own score bits bit-exact, metrics to 1e-12."""
    g = _load(golden_dir, "final_medium_d1024")
    dim, hidden, n_rows, n_imp, seed = (int(g[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    sd = syn.make_final_attention_state_dict(dim, hidden, seed=seed)
    assert sd_digest(sd) == str(g["sd_sha256"])
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand=str(g["cand"]), seed=seed + 3)
    ref_ranks = g["ranks"].astype(np.float64)
    assert np.array_equal(np.concatenate(oracle.rank_group_preds(g["scores"], imp.cand_len)), ref_ranks)
    grouped = oracle.group_items(ref_ranks, imp.cand_len)
    m = np.array([oracle.score_row(imp.labels[i], grouped[i]) for i in range(n_imp)])
    # exactly tied scores with different labels depend on numpy's unstable argsort (DESIGN section 1): AUC always
    tied = np.array([len(np.unique(r)) < len(r) for r in grouped])
    np.testing.assert_allclose(m[~tied], g["metrics"][~tied], atol=1e-12, rtol=0)
    np.testing.assert_allclose(m[:, 0], g["metrics"][:, 0], atol=1e-12, rtol=0)
    sub = slice(0, 64)  # the fp64 oracle on the first 64 impressions (the per-slot MLP is slow on the CPU)
    h_off, c_off = syn.csr_offsets(imp.hist_len), syn.csr_offsets(imp.cand_len)
    out = oracle.final_second_attention_score(sd, table, imp.hist_idx[:h_off[64]], imp.hist_len[sub],
                                              imp.cand_idx[:c_off[64]], imp.cand_len[sub], dtype=torch.float64)
    np.testing.assert_allclose(out["scores"], g["scores"][:c_off[64]], atol=2e-6, rtol=0)
    np.testing.assert_allclose(out["user"].float().numpy()[:32], g["user"], atol=3e-6, rtol=1e-5)


def test_latent_user_encoder_long_history_matches_reference(golden_dir):
    """BASELINE configs[4] shape (d=1024, 1024 latents, histories up to 200) through
    get_final_second_attention_score with LatentAttentionModel as the user encoder."""
    g = _load(golden_dir, "latent_user_cfg5_d1024_L1024_H200")
    dim, L, n_rows, n_imp, h_max, seed = (int(g[k]) for k in ("dim", "L", "n_rows", "n_imp", "h_max", "seed"))
    sd = syn.make_latent_state_dict(dim, L, seed=seed)
    assert sd_digest(sd) == str(g["sd_sha256"])
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_long_history_impressions(n_imp, n_rows, h_max, seed + 3)
    assert np.array_equal(imp.hist_len, g["hist_len"]) and int(imp.hist_len.max()) == h_max == 200
    out = oracle.latent_second_attention_score(sd, table, imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len,
                                               dtype=torch.float64, batch=5)
    np.testing.assert_allclose(out["user"].float().numpy(), g["user"], atol=2e-6, rtol=0)
    np.testing.assert_allclose(out["scores"], g["scores"], atol=2e-6, rtol=0)
    assert np.array_equal(np.concatenate(oracle.rank_group_preds(g["scores"], imp.cand_len)), g["ranks"])
    grouped = oracle.group_items(g["ranks"], imp.cand_len)
    m = np.array([oracle.score_row(imp.labels[i], grouped[i]) for i in range(n_imp)])
    np.testing.assert_allclose(m, g["metrics"], atol=1e-12, rtol=0)


def test_separable_rows_equal_padded_forward():
    """FinalAttention is separable per table row (SURVEY 8a row a9)."""
    sd = syn.make_final_attention_state_dict(32, 64, seed=3)
    table = syn.make_table(50, 32, seed=4)
    imp = syn.make_impressions(9, 50, h_max=7, seed=5)
    u = oracle.user_vectors(sd, table, imp.hist_idx, imp.hist_len, batch=4)
    X, Wl = oracle.final_attention_rows(sd, table)
    E = torch.exp(Wl)
    off = syn.csr_offsets(imp.hist_len)
    for i in range(imp.n):
        r = torch.from_numpy(imp.hist_idx[off[i]:off[i + 1]]).long()
        ui = (X[r] * E[r]).sum(0) / (E[r].sum(0) + 1e-10)
        torch.testing.assert_close(ui, u[i], atol=1e-12, rtol=1e-10)


def test_small_cases(golden_dir):
    g = _load(golden_dir, "small_cases")
    t = torch.Generator().manual_seed(7)
    table = torch.randn(11, 8, generator=t)
    groups = [np.array([3, 1, 4], dtype=np.int32), np.array([10], dtype=np.int32),
              np.array([0, 0, 5, 9, 2], dtype=np.int32), np.array([7, 8], dtype=np.int32)]
    emb, msk = oracle.final_attention_eval_collate(groups, table)
    assert np.array_equal(emb.numpy(), g["collate_emb"])
    assert np.array_equal(msk.numpy(), g["collate_mask"]) and msk.dtype == torch.int32
    ranks = np.concatenate(oracle.rank_group_preds(g["rank_scores"], g["rank_counts"]))
    assert np.array_equal(ranks, g["rank_out"], equal_nan=True)
    impressions = ["N1-0 N2-1 N3-0", "N2-0 N4-1", "N5-1 N1-0 N6-0 N7-0"]
    history = ["N9 N1 N8", "N8", "N4 N9 N10 N2"]
    sp = oracle.split_impressions_and_history(impressions, history)
    assert list(sp["news_list"]) == list(g["split_news"])
    for a, b in (("impression_rev_ind_array", "split_imp"), ("impression_len_list", "split_imp_len"),
                 ("history_rev_ind_array", "split_hist"), ("history_len_list", "split_hist_len")):
        assert np.array_equal(sp[a], g[b]) and sp[a].dtype == np.int32
    lab = np.array([list(l) + [-1] * (4 - len(l)) for l in sp["labels"]])
    assert np.array_equal(lab, g["split_labels"])


def test_oracle_against_live_reference_if_present():
    from oracle import ref_harness
    if not ref_harness.reference_available():
        pytest.skip("/root/reference not present (GPU box)")
    ref = ref_harness.load_reference(batch_size=16)
    model = ref_harness.make_reference_latent_model(ref, 256, 32, seed=11)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    x, mask = syn.make_token_batch(3, 9, 256, seed=12, min_len=1)
    with torch.no_grad():
        want = model(x, mask)
    got = oracle.latent_pool(sd, x, mask, dtype=torch.float32)
    torch.testing.assert_close(got, want, atol=2e-6, rtol=0)


def _new_attention_fixture(golden_dir):
    g = _load(golden_dir, "new_attention_d256")
    dim = int(g["dim"])
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w::")}
    table = syn.make_table(300, dim, seed=78)
    imp = syn.make_impressions(21, 300, h_max=12, seed=79)
    emb, msk = oracle.final_attention_eval_collate(oracle.group_items(imp.hist_idx, imp.hist_len), table)
    return g, sd, emb, msk, table, imp


def test_new_attention_matches_reference(golden_dir):
    g, sd, emb, msk, _, _ = _new_attention_fixture(golden_dir)
    out = oracle.new_attention(sd, emb, msk, num_layers=1, dtype=torch.float64).float().numpy()
    np.testing.assert_allclose(out, g["out"], atol=3e-6, rtol=1e-5)


def _final_score_fixture(golden_dir):
    g = _load(golden_dir, "final_score_blend_d256")
    dim, hidden, n_rows, n_imp, seed = (int(g[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    head_sd = {k[6:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("head::")}
    attn_sd = syn.make_final_attention_state_dict(dim, hidden, seed=seed)
    table = syn.make_table(n_rows, dim, seed=seed + 1)
    imp = syn.make_impressions(n_imp, n_rows, h_max=20, cand="small", seed=seed + 2)
    hb = g["history_bool"]
    h_off = syn.csr_offsets(imp.hist_len)
    hist_idx = np.concatenate([imp.hist_idx[h_off[i]:h_off[i + 1]] for i in range(n_imp) if hb[i]])
    return g, head_sd, attn_sd, table, imp, hb, hist_idx, imp.hist_len[hb]


def test_final_score_blend_matches_reference(golden_dir):
    g, head_sd, attn_sd, table, imp, hb, hist_idx, hist_len = _final_score_fixture(golden_dir)
    cls = oracle.classification_head(head_sd, table).squeeze(-1).numpy()
    np.testing.assert_allclose(cls, g["classification"], atol=2e-6, rtol=1e-5)
    out = oracle.final_score(attn_sd, table, hist_idx, hist_len, imp.cand_idx, imp.cand_len, hb, g["classification"],
                             alpha_param=0.7)
    np.testing.assert_allclose(out["scores"], g["scores"], atol=2e-6, rtol=0)
    assert np.array_equal(np.concatenate(oracle.rank_group_preds(g["scores"], imp.cand_len)), g["ranks"])


def test_dense_rank_and_auc_against_the_third_party_functions():
    """The arithmetic of the ranking / metric rows lives in un-pinned third-party code (SURVEY 8c): check the
    oracle's restatements against scipy.stats.rankdata and sklearn.roc_auc_score themselves on random groups
    with heavy ties, +-0, infinities and NaN (data_utils.py:414-415, evaluation.py:49)."""
    scipy_stats = pytest.importorskip("scipy.stats")
    metrics = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(2024)
    for trial in range(300):
        n = int(rng.integers(1, 80))
        kind = trial % 4
        if kind == 0:
            x = rng.standard_normal(n).astype(np.float32)
        elif kind == 1:
            x = (rng.integers(-3, 4, size=n) / 4.0).astype(np.float32)  # heavy ties, +0 / -0 below
            x[x == 0] *= rng.choice([-1.0, 1.0], size=int((x == 0).sum())).astype(np.float32)
        elif kind == 2:
            x = rng.standard_normal(n).astype(np.float32)
            x[rng.integers(0, n)] = np.inf
            x[rng.integers(0, n)] = -np.inf
        else:
            x = rng.standard_normal(n).astype(np.float32)
            x[rng.integers(0, n)] = np.nan
        want = scipy_stats.rankdata(-x, method="dense")
        got = oracle.dense_rank_desc(x)
        assert np.array_equal(np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64), equal_nan=True)
        if kind in (0, 1) and n >= 2:
            labels = rng.integers(0, 2, size=n)
            labels[0], labels[1] = 0, 1
            ranks = oracle.dense_rank_desc(x)
            assert abs(oracle._auc_tie_aware(labels, 1.0 / ranks) - metrics.roc_auc_score(labels, 1.0 / ranks)) <= 1e-12
