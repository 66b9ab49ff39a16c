"""GPU parity through the reference-named drop-in API (the calls scripts/eval.py makes)."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from news_recommendation_project_v2_b200 import synthetic as syn

pytestmark = pytest.mark.gpu


def _final_model(dim, hidden, seed, precision):
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention
    m = FinalAttention(dim, hidden, precision=precision)
    m.load_state_dict(syn.make_final_attention_state_dict(dim, hidden, seed=seed), strict=True)
    return m.eval()


def _rank_mismatches(got_ranks, ref_ranks, ref_scores, cand_len, gap):
    """Impressions whose dense ranks differ although every adjacent reference score gap exceeds `gap`."""
    off = syn.csr_offsets(cand_len)
    hard, soft = 0, 0
    for i in range(len(cand_len)):
        a, b = got_ranks[off[i]:off[i + 1]], ref_ranks[off[i]:off[i + 1]]
        if np.array_equal(a, b):
            continue
        s = np.sort(ref_scores[off[i]:off[i + 1]].astype(np.float64))
        if len(s) > 1 and np.min(np.diff(s)) <= gap:
            soft += 1
        else:
            hard += 1
    return hard, soft


@pytest.mark.parametrize("precision", ["fp32", "fp32x3"])
@pytest.mark.parametrize("name", ["final_small_d768", "final_large_d1024"])
def test_final_second_attention_score_fp32_matches_reference(golden_dir, name, precision):
    """fp32 path vs the reference's own outputs: scores 1e-5, rankings bit-exact wherever the
    reference's adjacent score gaps exceed 1e-5, metrics equal to 4 decimals.  "fp32x3" = the same fp32 tables with
    the row transform on the tensor cores as split-bf16 GEMMs (three hi/lo products accumulated in fp32): held to the
    same bars."""
    from news_recommendation_project_v2_b200.data_model_helper import (
        get_final_second_attention_score, get_final_attention_eval, get_cos_sim_scores)
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    dim, hidden, n_rows, n_imp, seed = (int(g[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    model = _final_model(dim, hidden, seed, precision)
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand=str(g["cand"]), seed=seed + 3)
    hb = np.ones(n_imp, dtype=bool)
    out = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, hb, model,
                                           precision=precision)
    assert out["scores"].dtype == np.float32 and out["scores"].shape == g["scores"].shape
    print(f"{name} {precision}: max |score - reference| = {np.abs(out['scores'] - g['scores']).max():.3e}")
    np.testing.assert_allclose(out["scores"], g["scores"], atol=1e-5, rtol=0)
    assert out["grouped_scores"].dtype == object and len(out["grouped_scores"]) == n_imp
    ranks = np.concatenate([np.asarray(r) for r in out["grouped_scores"]])
    hard, soft = _rank_mismatches(ranks, g["ranks"], g["scores"], imp.cand_len, gap=1e-5)
    assert hard == 0 and soft <= 2
    metrics = np.array([oracle.score_row(imp.labels[i], out["grouped_scores"][i]) for i in range(n_imp)])
    np.testing.assert_allclose(metrics.mean(0), g["metrics"].mean(0), atol=5e-5, rtol=0)
    user = get_final_attention_eval(imp.hist_idx, imp.hist_len, table, model, precision=precision)
    np.testing.assert_allclose(user.numpy(), g["user"], atol=2e-5, rtol=2e-5)
    sc = get_cos_sim_scores(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, model, precision=precision)
    assert sc.device.type == "cpu" and np.array_equal(sc.numpy(), out["scores"])


@pytest.mark.parametrize("precision", ["fp32", "fp32x3"])
def test_rank_exactness_on_1024_reference_impressions(golden_dir, precision):
    """1,024 impressions / 39,226 candidates scored by the UNMODIFIED reference (`final_medium_d1024`): scores within
    1e-5, every impression whose reference score gaps all exceed 1e-5 ranked bit-exactly, metric means to 4 decimals;
    the bf16 path is held to the metric bar on the same fixture."""
    from news_recommendation_project_v2_b200.data_model_helper import get_final_second_attention_score
    g = np.load(os.path.join(golden_dir, "final_medium_d1024.npz"))
    dim, hidden, n_rows, n_imp, seed = (int(g[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand=str(g["cand"]), seed=seed + 3)
    hb = np.ones(n_imp, dtype=bool)
    ref_ranks = g["ranks"].astype(np.float64)
    out = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, hb,
                                           _final_model(dim, hidden, seed, precision), precision=precision)
    np.testing.assert_allclose(out["scores"], g["scores"], atol=1e-5, rtol=0)
    ranks = np.concatenate([np.asarray(r) for r in out["grouped_scores"]])
    hard, soft = _rank_mismatches(ranks, ref_ranks, g["scores"], imp.cand_len, gap=1e-5)
    print(f"{precision}: {int((ranks != ref_ranks).sum())} of {len(ranks)} candidate ranks differ "
          f"({soft} impressions, all inside a 1e-5 score gap)")
    assert hard == 0 and soft <= 40
    metrics = np.array([oracle.score_row(imp.labels[i], out["grouped_scores"][i]) for i in range(n_imp)])
    np.testing.assert_allclose(metrics.mean(0), g["metrics"].mean(0), atol=5e-5, rtol=0)
    if precision == "fp32":
        b16 = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, hb,
                                               _final_model(dim, hidden, seed, "bf16"), precision="bf16")
        np.testing.assert_allclose(b16["scores"], g["scores"], atol=3e-3, rtol=0)
        rb = np.concatenate([np.asarray(r) for r in b16["grouped_scores"]])
        hard16, _ = _rank_mismatches(rb, ref_ranks, g["scores"], imp.cand_len, gap=6e-3)
        assert hard16 == 0
        mb = np.array([oracle.score_row(imp.labels[i], b16["grouped_scores"][i]) for i in range(n_imp)])
        # 1,024 impressions: a single swapped pair moves a mean by ~1e-3 / 1024; the 4-decimal bar is asserted on the
        # 2.4 M-impression workload (test_gpu_fullsize.py), here the means must agree to 1e-3
        np.testing.assert_allclose(mb.mean(0), g["metrics"].mean(0), atol=1e-3, rtol=0)


def test_final_second_attention_score_bf16(golden_dir):
    """bf16 throughput path: scores within 3e-3 of the fp32 reference (the reference's own bf16
    drift is 7.4e-4, BASELINE.md); ranks exact wherever reference gaps exceed 2x that tolerance."""
    from news_recommendation_project_v2_b200.data_model_helper import get_final_second_attention_score
    g = np.load(os.path.join(golden_dir, "final_large_d1024.npz"))
    dim, hidden, n_rows, n_imp, seed = (int(g[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    model = _final_model(dim, hidden, seed, "bf16")
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand="large", seed=seed + 3)
    out = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table,
                                           np.ones(n_imp, dtype=bool), model, precision="bf16")
    np.testing.assert_allclose(out["scores"], g["scores"], atol=3e-3, rtol=0)
    ranks = np.concatenate([np.asarray(r) for r in out["grouped_scores"]])
    hard, _ = _rank_mismatches(ranks, g["ranks"], g["scores"], imp.cand_len, gap=6e-3)
    assert hard == 0


@pytest.mark.parametrize("precision,tol_user,tol_score", [("fp32", 3e-6, 1e-5), ("bf16", 2e-3, 3e-3)])
def test_latent_user_encoder_long_history_matches_reference(golden_dir, precision, tol_user, tol_score):
    """BASELINE configs[4] shape end to end: LatentAttentionModel (d=1024, 1024 latents -> a softmax row spans a
    4-CTA cluster in the bf16 path) as the USER encoder, histories up to 200, through the widest seam
    (get_final_second_attention_score) against the reference's own outputs."""
    from news_recommendation_project_v2_b200.data_model_helper import (get_final_attention_eval,
                                                                       get_final_second_attention_score)
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    g = np.load(os.path.join(golden_dir, "latent_user_cfg5_d1024_L1024_H200.npz"))
    dim, L, n_rows, n_imp, h_max, seed = (int(g[k]) for k in ("dim", "L", "n_rows", "n_imp", "h_max", "seed"))
    model = LatentAttentionModel(dim=dim, num_latents=L, precision=precision).eval()
    model.load_state_dict(syn.make_latent_state_dict(dim, L, seed=seed), strict=True)
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_long_history_impressions(n_imp, n_rows, h_max, seed + 3)
    assert int(imp.hist_len.max()) == 200
    out = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table,
                                           np.ones(n_imp, dtype=bool), model, precision=precision)
    np.testing.assert_allclose(out["scores"], g["scores"], atol=tol_score, rtol=0)
    user = get_final_attention_eval(imp.hist_idx, imp.hist_len, table, model, precision=precision)
    np.testing.assert_allclose(user.numpy(), g["user"], atol=tol_user, rtol=0)
    ranks = np.concatenate([np.asarray(r) for r in out["grouped_scores"]])
    hard, soft = _rank_mismatches(ranks, g["ranks"], g["scores"], imp.cand_len, gap=2 * tol_score)
    assert hard == 0
    if precision == "fp32":
        assert soft <= 1
        metrics = np.array([oracle.score_row(imp.labels[i], out["grouped_scores"][i]) for i in range(n_imp)])
        np.testing.assert_allclose(metrics.mean(0), g["metrics"].mean(0), atol=5e-5, rtol=0)


def test_checkpoint_round_trip_through_factories_and_dataloader(golden_dir, tmp_path, monkeypatch):
    """The loader seams of the reference (modeling_utils.py:151-155, 274-279, 402-417 and the DataLoader of
    data_model_helper.py:122-130): state_dict written with torch.save -> get_*_model(path) (strict load,
    .to(DEVICE), eval) -> get_model_eval over a DataLoader with the reference's collate function."""
    from functools import partial

    from torch.utils.data import DataLoader

    from news_recommendation_project_v2_b200 import config, modeling_utils as mu
    from news_recommendation_project_v2_b200.data_utils import (FinalAttentionEvalDataset,
                                                                final_attention_eval_collate_fn)
    monkeypatch.setattr(config, "PRECISION", "fp32")
    # ---- FinalAttention: golden user vectors of the reference's get_final_attention_eval -------------
    g = np.load(os.path.join(golden_dir, "final_small_d768.npz"))
    dim, hidden, n_rows, n_imp, seed = (int(g[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    assert hidden == 4096  # the factory's fixed hidden size (modeling_utils.py:275)
    path = tmp_path / "Best_model_final_attention.pt"
    torch.save(syn.make_final_attention_state_dict(dim, hidden, seed=seed), path)
    monkeypatch.setattr(config, "REDUCED_DIM", dim)
    model = mu.get_final_attention_model(path)
    assert not model.training and next(model.parameters()).device.type == config.DEVICE.type == "cuda"
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand=str(g["cand"]), seed=seed + 3)
    loader = DataLoader(FinalAttentionEvalDataset(imp.hist_idx, imp.hist_len), batch_size=24, shuffle=False,
                        collate_fn=partial(final_attention_eval_collate_fn, news_embeddings=table), num_workers=0)
    user = mu.get_model_eval(loader, model)
    assert user.device.type == "cpu" and user.shape == (n_imp, dim)
    np.testing.assert_allclose(user.numpy(), g["user"], atol=2e-5, rtol=2e-5)
    with pytest.raises(RuntimeError):  # a checkpoint of another architecture must not load silently
        mu.get_final_attention_model(_save(tmp_path, {"linear1.weight": torch.zeros(3, 3)}))
    # ---- LatentAttentionModel at the reference's default dims (config.py:29-31; 64 latents) --------------
    g = np.load(os.path.join(golden_dir, "latent_default_d1024_L64.npz"))
    dim, L, B, S, seed = (int(g[k]) for k in ("dim", "L", "B", "S", "seed"))
    monkeypatch.setattr(config, "REDUCED_DIM", dim)
    monkeypatch.setattr(config, "EMBEDDING_DIM", dim)
    path = tmp_path / "Best_model_latent.pt"
    torch.save(syn.make_latent_state_dict(dim, L, seed=seed), path)
    lat = mu.get_latent_attention_model(path)
    assert sorted(lat.state_dict().keys()) == list(g["keys"])
    x, mask = syn.make_token_batch(B, S, dim, seed=seed + 1)
    loader = DataLoader(torch.utils.data.TensorDataset(x, mask), batch_size=3, shuffle=False)
    pooled = mu.get_model_eval(loader, lat)  # get_model_eval calls model(*batch) positionally (:411-414)
    np.testing.assert_allclose(pooled.numpy(), g["pooled"], atol=3e-6, rtol=0)


def _save(tmp_path, sd):
    p = tmp_path / "other.pt"
    torch.save(sd, p)
    return p


@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("bf16", 2e-2)])
def test_final_attention_module_forward(precision, tol):
    """FinalAttention.forward on a padded, masked batch (the DataLoader path of the reference)."""
    from news_recommendation_project_v2_b200.data_utils import final_attention_eval_collate_fn, group_items
    dim, hidden = 256, 512
    model = _final_model(dim, hidden, 31, precision)
    table = syn.make_table(300, dim, seed=32)
    imp = syn.make_impressions(19, 300, h_max=12, seed=33)
    groups = group_items(imp.hist_idx, imp.hist_len)
    emb, mask = final_attention_eval_collate_fn(list(groups), table)
    assert emb.device.type == "cpu" and mask.dtype == torch.int32
    want_e, want_m = oracle.final_attention_eval_collate(list(groups), table)
    assert torch.equal(emb, want_e) and torch.equal(mask, want_m)
    out = model(emb.cuda(), mask.cuda())
    want = oracle.final_attention(model.state_dict(), emb, mask)
    torch.testing.assert_close(out.cpu().double(), want, atol=tol, rtol=tol)
    with pytest.raises(Exception):
        model.train()(emb.cuda(), mask.cuda())
    model.eval()


def test_rank_group_preds_and_component(golden_dir):
    from news_recommendation_project_v2_b200.components import FinalAttentionComponent
    from news_recommendation_project_v2_b200.data_utils import rank_group_preds
    from news_recommendation_project_v2_b200.pipeline import Pipeline
    g = np.load(os.path.join(golden_dir, "small_cases.npz"))
    r = rank_group_preds(g["rank_scores"], g["rank_counts"])
    assert r.dtype == object
    assert np.array_equal(np.concatenate(list(r)), g["rank_out"], equal_nan=True)
    # pipeline seam: context_dict in, context_dict + {"scores","grouped_scores"} out (components.py:1013-1027)
    gf = np.load(os.path.join(golden_dir, "final_small_d768.npz"))
    dim, hidden, n_rows, n_imp, seed = (int(gf[k]) for k in ("dim", "hidden", "n_rows", "n_imp", "seed"))
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand="small", seed=seed + 3)
    owner = lambda lens: np.repeat(np.arange(len(lens), dtype=np.int32), lens)
    ctx = {
        "news_embeddings": syn.make_table(n_rows, dim, seed=seed + 2),
        "impression_rev_ind_array": np.stack([imp.cand_idx, owner(imp.cand_len)]),
        "impression_len_list": imp.cand_len,
        "history_rev_ind_array": np.stack([imp.hist_idx, owner(imp.hist_len)]),
        "history_len_list": imp.hist_len,
        "history_bool": np.ones(n_imp, dtype=bool),
        "labels": imp.labels,
    }
    comp = FinalAttentionComponent(attention_model=_final_model(dim, hidden, seed, "fp32"), precision="fp32")
    out, _ = Pipeline("eval", [("final_attn_comp", comp)]).transform(ctx)
    np.testing.assert_allclose(out["scores"], gf["scores"], atol=1e-5, rtol=0)
    assert "labels" in out and len(out["grouped_scores"]) == n_imp
    with pytest.raises(AssertionError):
        comp.transform({k: v for k, v in ctx.items() if k != "history_bool"})


def test_latent_model_as_user_encoder():
    """LatentAttentionModel shares the (embeddings, mask) contract (components.py:504,675):
    per-row transform + mean-pool + L2 normalise, then the same cosine / rank path."""
    from news_recommendation_project_v2_b200.data_model_helper import get_final_second_attention_score
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    dim, L = 256, 32
    m = LatentAttentionModel(dim=dim, num_latents=L, heads=2, dim_head=64, precision="fp32").eval()
    m.load_state_dict(syn.make_latent_state_dict(dim, L, heads=2, dim_head=64, seed=41))
    table = syn.make_table(400, dim, seed=42)
    imp = syn.make_impressions(23, 400, h_max=9, seed=43)
    out = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table,
                                           np.ones(23, dtype=bool), m, precision="fp32")
    groups = oracle.group_items(imp.hist_idx, imp.hist_len)
    emb, msk = oracle.final_attention_eval_collate(groups, table)
    u = oracle.latent_pool(m.state_dict(), emb, msk, heads=2, dim_head=64)
    want = oracle.cosine_scores(u, table, imp.cand_idx, imp.cand_len).numpy()
    np.testing.assert_allclose(out["scores"], want, atol=1e-5, rtol=0)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_streamed_engine_and_pipelined_host_scoring_match_resident_path(precision):
    """ScoringEngine(cache_table=False) + score_host (copy/compute/copy-out streams, impression chunks)
    must be bit-identical to the single-launch resident path."""
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    dim, hidden, n_rows, n_imp = 256, 512, 40000, 3000  # > 2 table chunks of 16384 rows
    model = _final_model(dim, hidden, 51, precision)
    table = syn.make_table(n_rows, dim, seed=52)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand="large", seed=53)
    ref_eng = ScoringEngine(table, model, precision=precision)
    _, want_s, want_r = ref_eng.score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len)
    eng = ScoringEngine(table.pin_memory(), model, precision=precision, cache_table=False)
    assert torch.equal(eng.hist_x, ref_eng.hist_x) and torch.equal(eng.hist_e, ref_eng.hist_e)
    assert torch.equal(eng.cand, ref_eng.cand)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    for n_chunks in (1, 3, 8):
        s, r = eng.score_host(t(imp.hist_idx), t(syn.csr_offsets(imp.hist_len)), t(imp.cand_idx),
                              t(syn.csr_offsets(imp.cand_len)), n_chunks=n_chunks)
        assert s.device.type == "cpu" and torch.equal(s, want_s.cpu()) and torch.equal(r, want_r.cpu())
    bad = imp.hist_idx.copy()
    bad[5] = n_rows + 3
    with pytest.raises(IndexError):
        eng.score_host(t(bad), t(syn.csr_offsets(imp.hist_len)), t(imp.cand_idx), t(syn.csr_offsets(imp.cand_len)))


def test_mind_metrics_kernel_matches_reference_golden(golden_dir):
    """nrb_mind_metrics vs evaluation.score_row outputs of the reference (AUC/MRR/nDCG to 1e-12)."""
    from news_recommendation_project_v2_b200 import ops
    from news_recommendation_project_v2_b200.evaluation import score
    for name in ("final_small_d768", "final_large_d1024"):
        g = np.load(os.path.join(golden_dir, name + ".npz"))
        n_rows, n_imp, seed = int(g["n_rows"]), int(g["n_imp"]), int(g["seed"])
        imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand=str(g["cand"]), seed=seed + 3)
        ranks = torch.from_numpy(g["ranks"].astype(np.int32)).cuda()
        labels = torch.from_numpy(np.concatenate([np.asarray(l, dtype=np.int8) for l in imp.labels])).cuda()
        off = torch.from_numpy(syn.csr_offsets(imp.cand_len)).cuda()
        per, sums = ops.mind_metrics(ranks, labels, off)
        per = per.cpu().numpy()
        # MRR / nDCG depend on the order among candidates with EXACTLY tied scores but different labels;
        # the reference takes that order from numpy's default (unstable, SIMD-dependent) argsort, so those
        # impressions are compared on AUC only (tie-order independent) -- 1 of 48 in this fixture.
        grouped = oracle.group_items(g["ranks"], imp.cand_len)
        discordant = np.array([any(len(set(np.asarray(imp.labels[i])[grouped[i] == v])) > 1
                                   for v in np.unique(grouped[i])) for i in range(n_imp)])
        np.testing.assert_allclose(per[~discordant], g["metrics"][~discordant], atol=1e-12, rtol=0)
        np.testing.assert_allclose(per[:, 0], g["metrics"][:, 0], atol=1e-12, rtol=0)
        assert discordant.sum() <= 2
        np.testing.assert_allclose(sums.cpu().numpy()[:4] / n_imp, per.mean(0), atol=1e-12, rtol=0)
        np.testing.assert_allclose(per.mean(0), g["metrics"].mean(0), atol=5e-5, rtol=0)  # 4-decimal bar
        d = score(grouped, imp.labels)
        assert d["num_samples"] == n_imp and abs(d["auc"] - g["metrics"][:, 0].mean()) < 1e-12
    # ties (reversed stable order), more than 512 candidates, single-class impression -> NaN / ValueError
    rng = np.random.default_rng(5)
    counts = np.array([7, 600, 40, 3], dtype=np.int32)
    ranks_l, labels_l = [], []
    for c in counts:
        sc = rng.integers(0, max(2, c // 3), size=c).astype(np.float32)  # heavy ties
        ranks_l.append(oracle.dense_rank_desc(sc))
        lab = (rng.random(c) < 0.3).astype(np.int8)
        lab[0], lab[1] = 1, 0
        labels_l.append(lab)
    labels_l[3][:] = 1  # single class
    per, sums = ops.mind_metrics(torch.from_numpy(np.concatenate(ranks_l).astype(np.int32)).cuda(),
                                 torch.from_numpy(np.concatenate(labels_l)).cuda(),
                                 torch.from_numpy(syn.csr_offsets(counts)).cuda())
    per = per.cpu().numpy()
    for i in range(3):
        y = labels_l[i].astype(np.float32)
        ys = 1.0 / ranks_l[i]
        order = np.argsort(ys, kind="stable")[::-1]
        ideal = np.argsort(y, kind="stable")[::-1]
        want_mrr = np.sum(np.take(y, order) / (np.arange(len(y)) + 1)) / y.sum()
        auc = oracle._auc_tie_aware(y, ys)
        assert abs(per[i, 0] - auc) < 1e-12 and abs(per[i, 1] - want_mrr) < 1e-12
        dcg = lambda o, k: np.sum((2.0 ** y[o[:k]] - 1) / np.log2(np.arange(len(o[:k])) + 2))
        assert abs(per[i, 2] - dcg(order, 5) / dcg(ideal, 5)) < 1e-12
        assert abs(per[i, 3] - dcg(order, 10) / dcg(ideal, 10)) < 1e-12
    assert np.isnan(per[3]).all() and int(sums[4].item()) == 3
    with pytest.raises(ValueError):
        score(ranks_l, labels_l)


def test_mind_metrics_kernel_several_impressions_per_warp():
    """nrb_mind_metrics with every warp of its grid (SMs x 16 CTAs x 8 warps) on >= 3 impressions, against the
    vectorised fp64 score_row (stable tie order): the `large` candidate counts plus 600 / 1,500 (global-memory path),
    heavy rank ties, label-2 gains, single-class, NaN-group and empty impressions next to ordinary ones on one warp."""
    from news_recommendation_project_v2_b200 import ops
    from tests import segment_oracle as so
    W = torch.cuda.get_device_properties(0).multi_processor_count * 16 * 8
    n_imp = 3 * W + W // 6
    assert n_imp // W >= 3 and n_imp >= 3 * W
    rng = np.random.default_rng(12)
    counts = np.clip(np.rint(rng.lognormal(np.log(30.0), 0.7, size=n_imp)), 2, 300).astype(np.int64)
    counts[[3, W + 7, 2 * W + 11]] = 600
    counts[[5, W + 9, 3 * W + 1]] = 1500
    empty, zero_rank, all_neg, all_pos = [W + 13, 2], [17, 2 * W + 17], [19, 2 * W + 3], [W + 21, 23]
    counts[empty] = 0
    off = so.csr(counts)
    n = int(off[-1])
    scores = rng.integers(0, 8, size=n).astype(np.float32)  # heavy ties: at most 8 distinct scores per impression
    scores[off[3]:off[4]] = rng.integers(0, 200, size=600)
    ranks, _ = so.dense_rank_segments(torch.from_numpy(scores), torch.from_numpy(off))
    ranks = ranks.numpy()
    labels = (rng.random(n) < 0.3).astype(np.int8)
    starts = off[:-1][counts > 0]
    labels[starts], labels[starts + 1] = 1, 0  # both classes
    two = rng.choice(n_imp, size=n_imp // 50, replace=False)
    two = np.union1d(two[counts[two] > 0], [0, W, 2 * W, 3])
    labels[off[two]] = 2  # gains 2^y - 1 = 3
    for i in zero_rank:
        ranks[off[i]:off[i + 1]] = 0  # a NaN group's sentinel
    for i, v in [(i, 0) for i in all_neg] + [(i, 1) for i in all_pos]:
        labels[off[i]:off[i + 1]] = v
    want = so.mind_metrics_segments(ranks, labels, counts)
    invalid = np.isnan(want[:, 0])
    assert np.array_equal(np.flatnonzero(invalid), np.sort(empty + zero_rank + all_neg + all_pos))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    per, sums = ops.mind_metrics(t(ranks), t(labels), t(off))
    per, sums = per.cpu().numpy(), sums.cpu().numpy()
    assert np.array_equal(np.isnan(per), np.isnan(want))
    np.testing.assert_allclose(per, want, atol=1e-12, rtol=0)
    print(f"\nmind metrics: {n_imp} impressions on {W} warps, max |err| {np.abs(per - want)[~invalid].max():.2e}")
    want_sums = want[~invalid].sum(0)
    # atomics in a varying order: 1e-9 relative
    np.testing.assert_allclose(sums[:4], want_sums, rtol=1e-9, atol=0)
    assert sums[4] == (~invalid).sum()
    none, sums2 = ops.mind_metrics(t(ranks), t(labels), t(off), want_per_impression=False)
    sums2 = sums2.cpu().numpy()
    assert none is None
    np.testing.assert_allclose(sums2[:4], want_sums, rtol=1e-9, atol=0)
    assert sums2[4] == (~invalid).sum()


@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("bf16", 3e-2)])
def test_new_attention_arm(golden_dir, precision, tol):
    """NewAttention (attention.py:209-279): LayerNorm chain + per-dimension exp pooling, module and engine."""
    from tests.test_oracle_golden import _new_attention_fixture
    from news_recommendation_project_v2_b200.attention import NewAttention
    from news_recommendation_project_v2_b200.data_model_helper import get_cos_sim_scores
    g, sd, emb, msk, table, imp = _new_attention_fixture(golden_dir)
    m = NewAttention(hidden_size=int(g["dim"]), num_hidden_layers=1, precision=precision).eval()
    assert sorted(m.state_dict().keys()) == list(g["keys"])  # dead attention / MLP weights kept for checkpoints
    assert [str(tuple(m.state_dict()[k].shape)) for k in sorted(m.state_dict())] == list(g["shapes"])
    m.load_state_dict(sd, strict=False)
    out = m(emb.cuda(), msk.cuda()).cpu().numpy()
    np.testing.assert_allclose(out, g["out"], atol=tol, rtol=tol)
    # engine path: per-row tables + fused score/rank
    sc = get_cos_sim_scores(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, m, precision=precision)
    u = oracle.new_attention(sd, emb, msk)
    want = oracle.cosine_scores(u, table, imp.cand_idx, imp.cand_len).numpy()
    np.testing.assert_allclose(sc.numpy(), want, atol=1e-5 if precision == "fp32" else 5e-3, rtol=0)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 4e-3)])
def test_final_score_blend_and_classification_head(golden_dir, precision, tol):
    """get_final_score (data_model_helper.py:272-301): classification baseline + cosine blended inside the fused
    score/rank kernel, no-history impressions fall back to the baseline."""
    from tests.test_oracle_golden import _final_score_fixture
    from news_recommendation_project_v2_b200.data_model_helper import (get_classification_preds, get_final_score,
                                                                       get_final_only_attention_score)
    from news_recommendation_project_v2_b200.modeling_utils import ClassificationHead, WeightedSumModel
    g, head_sd, attn_sd, table, imp, hb, hist_idx, hist_len = _final_score_fixture(golden_dir)
    dim, hidden = int(g["dim"]), int(g["hidden"])
    head = ClassificationHead(dim, dim, 1, precision=precision).eval()
    head.load_state_dict(head_sd, strict=True)
    cls = get_classification_preds(table, head)
    np.testing.assert_allclose(cls, g["classification"], atol=tol * 2, rtol=tol)
    attn = _final_model(dim, hidden, int(g["seed"]), precision)
    wsum = WeightedSumModel()
    with torch.no_grad():
        wsum.alpha.fill_(0.7)
    # feed the REFERENCE's baseline so that only the fused blend / cosine / rank are under test
    out = get_final_score(hist_idx, hist_len, imp.cand_idx, imp.cand_len, table, g["classification"], hb, attn, wsum,
                          precision=precision)
    np.testing.assert_allclose(out["scores"], g["scores"], atol=tol, rtol=0)
    ranks = np.concatenate([np.asarray(r) for r in out["grouped_scores"]])
    assert np.array_equal(ranks, np.concatenate(oracle.rank_group_preds(out["scores"], imp.cand_len)))
    if precision == "fp32":
        hard, soft = _rank_mismatches(ranks, g["ranks"], g["scores"], imp.cand_len, gap=1e-5)
        assert hard == 0 and soft <= 1
    # impressions without history carry the baseline bit for bit
    off = syn.csr_offsets(imp.cand_len)
    for i in np.flatnonzero(~hb):
        assert np.array_equal(out["scores"][off[i]:off[i + 1]], g["classification"][imp.cand_idx[off[i]:off[i + 1]]])
    only = get_final_only_attention_score(hist_idx, hist_len, imp.cand_idx, imp.cand_len, table, g["classification"],
                                          hb, attn, precision=precision)
    want = oracle.final_score(attn_sd, table, hist_idx, hist_len, imp.cand_idx, imp.cand_len, hb, g["classification"],
                              alpha_param=60.0)["scores"]  # sigmoid(60) == 1: pure cosine where there is history
    np.testing.assert_allclose(only["scores"], want, atol=tol, rtol=0)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 5e-3)])
def test_row_width_384_runs_on_zero_padded_tables(precision, tol):
    """Embedding widths that are not a multiple of 512 bytes (384: bge-small, reference config.py:63) go through
    zero-padded copies of the tables: same scores / ranks / user vectors as the oracle at the logical width, on the
    engine path, the pipelined host path, the module forward and the latent user encoder."""
    from news_recommendation_project_v2_b200.data_model_helper import get_final_second_attention_score
    from news_recommendation_project_v2_b200.data_utils import final_attention_eval_collate_fn, group_items
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    dim, hidden, n_rows, n_imp = 384, 512, 3000, 150
    model = _final_model(dim, hidden, 71, precision)
    table = syn.make_table(n_rows, dim, seed=72)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand="large", seed=73)
    ref = oracle.final_second_attention_score(model.state_dict(), table, imp.hist_idx, imp.hist_len, imp.cand_idx,
                                              imp.cand_len)
    out = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table,
                                           np.ones(n_imp, dtype=bool), model, precision=precision)
    np.testing.assert_allclose(out["scores"], ref["scores"], atol=tol, rtol=0)
    ranks = np.concatenate([np.asarray(r) for r in out["grouped_scores"]])
    assert np.array_equal(ranks, np.concatenate(oracle.rank_group_preds(out["scores"], imp.cand_len)))
    hard, _ = _rank_mismatches(ranks, np.concatenate(ref["grouped_scores"]), ref["scores"], imp.cand_len, 2 * tol)
    assert hard == 0
    # user vectors at the logical width; host pipeline == device path bit for bit
    eng = ScoringEngine(table, model, precision=precision)
    user, s_dev, r_dev = eng.score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, want_user=True)
    assert user.shape == (n_imp, dim) and eng.cand.shape == (n_rows, dim)
    want_u = oracle.user_vectors(model.state_dict(), table, imp.hist_idx, imp.hist_len)
    np.testing.assert_allclose(user.cpu().numpy(), want_u.float().numpy(), atol=2e-5 if precision == "fp32" else 2e-2, rtol=0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    s_h, r_h = eng.score_host(t(imp.hist_idx), t(syn.csr_offsets(imp.hist_len)), t(imp.cand_idx),
                              t(syn.csr_offsets(imp.cand_len)), n_chunks=3)
    assert torch.equal(s_h, s_dev.cpu()) and torch.equal(r_h, r_dev.cpu())
    # new weights on the SAME engine: the padded kernel copies must follow the rebuilt tables (which may well land
    # at the old addresses)
    with torch.no_grad():
        model.linear3.bias.add_(0.25)
    eng.prepare_user_encoder(eng.cand)
    _, s_new, r_new = eng.score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len)
    _, s_fresh, r_fresh = ScoringEngine(table, model, precision=precision).score(imp.hist_idx, imp.hist_len,
                                                                                 imp.cand_idx, imp.cand_len)
    assert torch.equal(s_new, s_fresh) and torch.equal(r_new, r_fresh) and not torch.equal(s_new, s_dev)
    # module forward on a padded, masked batch
    groups = group_items(imp.hist_idx[:int(imp.hist_len[:20].sum())], imp.hist_len[:20])
    emb, mask = final_attention_eval_collate_fn(list(groups), table)
    got = model(emb.cuda(), mask.cuda())
    want = oracle.final_attention(model.state_dict(), emb, mask)
    torch.testing.assert_close(got.cpu().double(), want, atol=2e-5 if precision == "fp32" else 2e-2, rtol=2e-2)
    # latent model as user encoder at the same width
    m = LatentAttentionModel(dim=dim, num_latents=32, heads=2, dim_head=64, precision=precision).eval()
    m.load_state_dict(syn.make_latent_state_dict(dim, 32, heads=2, dim_head=64, seed=74))
    out = get_final_second_attention_score(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table,
                                           np.ones(n_imp, dtype=bool), m, precision=precision)
    emb, msk = oracle.final_attention_eval_collate(oracle.group_items(imp.hist_idx, imp.hist_len), table)
    u = oracle.latent_pool(m.state_dict(), emb, msk, heads=2, dim_head=64)
    want = oracle.cosine_scores(u, table, imp.cand_idx, imp.cand_len).numpy()
    np.testing.assert_allclose(out["scores"], want, atol=tol, rtol=0)
