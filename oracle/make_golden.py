"""Mint golden vectors by running the UNMODIFIED reference in this container.

    python oracle/make_golden.py            # writes tests/golden/*.npz

TEST INFRASTRUCTURE.  Needs /root/reference (read-only); the GPU box never runs
this.  Inputs are regenerated at test time from the seeds recorded here through
`news_recommendation_project_v2_b200.synthetic`; only reference OUTPUTS (and a
checksum of the weights they were produced with) are stored, so the fixtures
stay small.
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np
import pandas as pd
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness  # noqa: E402
from news_recommendation_project_v2_b200 import synthetic as syn  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def sd_digest(sd: dict) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().contiguous().numpy().tobytes())
    return h.hexdigest()


def golden_latent(ref, name, dim, L, B, S, seed):
    model = ref_harness.make_reference_latent_model(ref, dim, L, seed=seed)
    sd = syn.make_latent_state_dict(dim, L, seed=seed)
    missing = model.load_state_dict(sd, strict=True)  # key compatibility (SURVEY 8a a1)
    assert not missing.missing_keys and not missing.unexpected_keys
    x, mask = syn.make_token_batch(B, S, dim, seed=seed + 1)
    with torch.no_grad():
        pooled = model(x, mask)
        unpooled0 = model(x[:1], None)[0]
    np.savez_compressed(
        os.path.join(GOLD, f"{name}.npz"),
        dim=dim, L=L, B=B, S=S, seed=seed, sd_sha256=sd_digest(sd),
        pooled=pooled.numpy(), unpooled0=unpooled0.numpy(),
        keys=np.array(sorted(model.state_dict().keys())),
        shapes=np.array([str(tuple(model.state_dict()[k].shape)) for k in sorted(model.state_dict().keys())]),
    )
    print(name, pooled.shape, float(pooled.norm(dim=-1).mean()))


def golden_latent_short_masks(ref):
    """d=256, 32 latents, token masks as short as one token (min_len=1: lengths 6, 6, 4), pooled by the reference;
    plus the digests of d=256 checkpoints (FinalAttention hidden 4096, LatentAttentionModel 64 latents) that the
    reference's modules load strictly, for the checkpoint-factory test."""
    dim, L, seed = 256, 32, 11
    model = ref_harness.make_reference_latent_model(ref, dim, L, seed=seed)
    sd = syn.make_latent_state_dict(dim, L, seed=seed)
    model.load_state_dict(sd, strict=True)
    x, mask = syn.make_token_batch(3, 9, dim, seed=12, min_len=1)
    with torch.no_grad():
        pooled = model(x, mask)
    fa_sd = syn.make_final_attention_state_dict(dim, 4096, seed=dim)
    ref_harness.make_reference_final_attention(ref, dim, 4096, seed=dim).load_state_dict(fa_sd, strict=True)
    lat_sd = syn.make_latent_state_dict(dim, 64, seed=dim + 1)
    ref_harness.make_reference_latent_model(ref, dim, 64, seed=dim + 1).load_state_dict(lat_sd, strict=True)
    np.savez_compressed(
        os.path.join(GOLD, "latent_short_masks_d256_L32.npz"),
        dim=dim, L=L, seed=seed, sd_sha256=sd_digest(sd), mask_len=mask.sum(1).numpy(), pooled=pooled.numpy(),
        final_attention_h4096_sha256=sd_digest(fa_sd), latent_L64_sha256=sd_digest(lat_sd),
    )
    print("latent_short_masks_d256_L32", pooled.shape, mask.sum(1).tolist())


def golden_final(ref, name, dim, hidden, n_rows, n_imp, cand, seed, users_kept=None):
    model = ref_harness.make_reference_final_attention(ref, dim, hidden, seed=seed)
    sd = syn.make_final_attention_state_dict(dim, hidden, seed=seed)
    model.load_state_dict(sd, strict=True)
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_impressions(n_imp, n_rows, h_max=50, cand=cand, seed=seed + 3)
    dmh = ref.data_model_helper
    hb = pd.Series(np.ones(n_imp, dtype=bool))
    with torch.no_grad():
        out = dmh.get_final_second_attention_score(
            imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, hb, model)
        user = dmh.get_final_attention_eval(imp.hist_idx, imp.hist_len, table, model)
    ranks = np.concatenate([np.asarray(r, dtype=np.float64) for r in out["grouped_scores"]])
    metrics = np.array([ref.evaluation.score_row((imp.labels[i], out["grouped_scores"][i], i))
                        for i in range(n_imp)], dtype=np.float64)
    np.savez_compressed(
        os.path.join(GOLD, f"{name}.npz"),
        dim=dim, hidden=hidden, n_rows=n_rows, n_imp=n_imp, cand=cand, seed=seed,
        sd_sha256=sd_digest(sd), scores=np.asarray(out["scores"], dtype=np.float32),
        ranks=ranks if users_kept is None else ranks.astype(np.int16),  # medium fixture: compact storage
        user=user.numpy() if users_kept is None else user.numpy()[:users_kept], metrics=metrics,
    )
    print(name, "scores", out["scores"].shape, "mean metrics", metrics.mean(axis=0))


def golden_latent_user_encoder(ref, name, dim, L, n_rows, n_imp, h_max, seed):
    """BASELINE configs[4] shape: LatentAttentionModel as the USER encoder (latent_attention.py:134-171) driven
    through get_final_second_attention_score (data_model_helper.py:416-443) with histories up to h_max."""
    model = ref_harness.make_reference_latent_model(ref, dim, L, seed=seed)
    sd = syn.make_latent_state_dict(dim, L, seed=seed)
    model.load_state_dict(sd, strict=True)
    table = syn.make_table(n_rows, dim, seed=seed + 2)
    imp = syn.make_long_history_impressions(n_imp, n_rows, h_max, seed + 3)
    dmh = ref.data_model_helper
    hb = pd.Series(np.ones(n_imp, dtype=bool))
    with torch.no_grad():
        out = dmh.get_final_second_attention_score(
            imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, hb, model)
        user = dmh.get_final_attention_eval(imp.hist_idx, imp.hist_len, table, model)
    ranks = np.concatenate([np.asarray(r, dtype=np.float64) for r in out["grouped_scores"]])
    metrics = np.array([ref.evaluation.score_row((imp.labels[i], out["grouped_scores"][i], i))
                        for i in range(n_imp)], dtype=np.float64)
    np.savez_compressed(
        os.path.join(GOLD, f"{name}.npz"),
        dim=dim, L=L, n_rows=n_rows, n_imp=n_imp, h_max=h_max, seed=seed, sd_sha256=sd_digest(sd),
        hist_len=imp.hist_len, scores=np.asarray(out["scores"], dtype=np.float32), ranks=ranks,
        user=user.numpy(), metrics=metrics,
    )
    print(name, "scores", out["scores"].shape, "max H", int(imp.hist_len.max()), "mean metrics", metrics.mean(axis=0))


def golden_new_attention(ref):
    """NewAttention (attention.py:209-279) forward on a padded batch; weights = the reference's own seeded init
    (LayerNorm affine perturbed so it is exercised), stored because the key set is large and mostly dead."""
    import news_rec_utils.attention as att
    dim = 256
    torch.manual_seed(77)
    model = att.NewAttention(hidden_size=dim, num_hidden_layers=1).eval()
    with torch.no_grad():
        ln = model.encoder.layer[0].g_mlp_layernorm
        ln.weight.add_(0.1 * torch.randn(dim))
        ln.bias.add_(0.1 * torch.randn(dim))
    table = syn.make_table(300, dim, seed=78)
    imp = syn.make_impressions(21, 300, h_max=12, seed=79)
    emb, msk = ref.data_utils.final_attention_eval_collate_fn(list(ref.data_utils.group_items(imp.hist_idx, imp.hist_len)), table)
    with torch.no_grad():
        out = model(emb, msk)
    live = {k: v.numpy() for k, v in model.state_dict().items() if "g_mlp_layernorm" in k or k.startswith("linear1")}
    np.savez_compressed(os.path.join(GOLD, "new_attention_d256.npz"), dim=dim, out=out.numpy(),
                        keys=np.array(sorted(model.state_dict().keys())),
                        shapes=np.array([str(tuple(model.state_dict()[k].shape)) for k in sorted(model.state_dict().keys())]),
                        **{"w::" + k: v for k, v in live.items()})
    print("new_attention", out.shape)


def golden_final_score(ref):
    """get_final_score (data_model_helper.py:272-301): ClassificationHead baseline + FinalAttention cosine blended by
    WeightedSumModel, with a mix of impressions with / without history."""
    dim, hidden, n_rows, n_imp, seed = 256, 512, 1500, 40, 321
    mu, dmh = ref.modeling_utils, ref.data_model_helper
    torch.manual_seed(seed)
    head = mu.ClassificationHead(in_dim=dim, hidden_dim=dim, out_dim=1).eval()
    attn = ref_harness.make_reference_final_attention(ref, dim, hidden, seed=seed)
    attn.load_state_dict(syn.make_final_attention_state_dict(dim, hidden, seed=seed))
    wsum = mu.WeightedSumModel()
    with torch.no_grad():
        wsum.alpha.fill_(0.7)
    table = syn.make_table(n_rows, dim, seed=seed + 1)
    imp = syn.make_impressions(n_imp, n_rows, h_max=20, cand="small", seed=seed + 2)
    hb = np.ones(n_imp, dtype=bool)
    hb[[3, 4, 17, 30]] = False
    h_off = syn.csr_offsets(imp.hist_len)
    hist_idx = np.concatenate([imp.hist_idx[h_off[i]:h_off[i + 1]] for i in range(n_imp) if hb[i]])
    hist_len = imp.hist_len[hb]
    with torch.no_grad():
        cls = dmh.get_classification_preds(table, head)
        out = dmh.get_final_score(hist_idx, hist_len, imp.cand_idx, imp.cand_len, table, cls, pd.Series(hb), attn, wsum)
    np.savez_compressed(os.path.join(GOLD, "final_score_blend_d256.npz"), dim=dim, hidden=hidden, n_rows=n_rows,
                        n_imp=n_imp, seed=seed, history_bool=hb, classification=cls.astype(np.float32),
                        scores=np.asarray(out["scores"], dtype=np.float32),
                        ranks=np.concatenate([np.asarray(r, dtype=np.float64) for r in out["grouped_scores"]]),
                        **{"head::" + k: v.numpy() for k, v in head.state_dict().items()})
    print("final_score_blend", out["scores"].shape)


def golden_small(ref):
    du = ref.data_utils
    # collate (data_utils.py:784-791)
    g = torch.Generator().manual_seed(7)
    table = torch.randn(11, 8, generator=g)
    groups = [np.array([3, 1, 4], dtype=np.int32), np.array([10], dtype=np.int32),
              np.array([0, 0, 5, 9, 2], dtype=np.int32), np.array([7, 8], dtype=np.int32)]
    emb, msk = du.final_attention_eval_collate_fn(groups, table)
    # dense rank (data_utils.py:414-415) with ties, +-0 and a NaN group
    scores = np.array([0.5, 0.25, 0.5, -1.0, 0.0, -0.0, 3.0, 1e-9, 2.0, 2.0, 2.0, 1.0, np.nan, 0.3, 7.0],
                      dtype=np.float32)
    counts = np.array([4, 4, 3, 1, 3], dtype=np.int32)
    ranks = du.rank_group_preds(scores, counts)
    ranks_flat = np.concatenate([np.asarray(r, dtype=np.float64) for r in ranks])
    # split (data_utils.py:168-232)
    impressions = ["N1-0 N2-1 N3-0", "N2-0 N4-1", "N5-1 N1-0 N6-0 N7-0"]
    history = ["N9 N1 N8", "N8", "N4 N9 N10 N2"]
    sp = du.split_impressions_and_history(impressions, history)
    np.savez_compressed(
        os.path.join(GOLD, "small_cases.npz"),
        collate_emb=emb.numpy(), collate_mask=msk.numpy(),
        rank_scores=scores, rank_counts=counts, rank_out=ranks_flat,
        split_news=sp["news_list"], split_imp=sp["impression_rev_ind_array"],
        split_imp_len=sp["impression_len_list"], split_hist=sp["history_rev_ind_array"],
        split_hist_len=sp["history_len_list"],
        split_labels=np.array([list(l) + [-1] * (4 - len(l)) for l in sp["labels"]]),
    )
    print("small cases ok", ranks_flat)


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    ref = ref_harness.load_reference(batch_size=16)
    only = set(sys.argv[1:])  # optional: names of the fixtures to (re)generate
    if only:
        if "latent_cfg5_d1024_L1024" in only:
            golden_latent(ref, "latent_cfg5_d1024_L1024", 1024, 1024, 4, 24, seed=555)
        if "final_medium_d1024" in only:
            golden_final(ref, "final_medium_d1024", 1024, 4096, 20000, 1024, "large", seed=7, users_kept=32)
        if "latent_user_cfg5_d1024_L1024_H200" in only:
            golden_latent_user_encoder(ref, "latent_user_cfg5_d1024_L1024_H200", 1024, 1024, 3000, 20, 200, seed=777)
        if "latent_short_masks_d256_L32" in only:
            golden_latent_short_masks(ref)
        return
    golden_small(ref)
    golden_new_attention(ref)
    golden_final_score(ref)
    golden_latent(ref, "latent_cfg1_d768_L512", 768, 512, 32, 64, seed=1234)
    golden_latent(ref, "latent_default_d1024_L64", 1024, 64, 4, 16, seed=4321)
    golden_final(ref, "final_small_d768", 768, 4096, 4096, 64, "small", seed=1234)
    golden_final(ref, "final_large_d1024", 1024, 4096, 2048, 48, "large", seed=99)
    # 1,024 impressions / 37 k candidates through the unmodified reference: the rank-exactness fixture
    golden_final(ref, "final_medium_d1024", 1024, 4096, 20000, 1024, "large", seed=7, users_kept=32)
    # BASELINE configs[4] shapes (d=1024, 1024 latents, histories up to 200)
    golden_latent(ref, "latent_cfg5_d1024_L1024", 1024, 1024, 4, 24, seed=555)
    golden_latent_user_encoder(ref, "latent_user_cfg5_d1024_L1024_H200", 1024, 1024, 3000, 20, 200, seed=777)
    golden_latent_short_masks(ref)


if __name__ == "__main__":
    main()
