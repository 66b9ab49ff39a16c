"""Drop-in scoring seams (reference: news_rec_utils/data_model_helper.py).

  get_final_attention_eval            data_model_helper.py:112-131
  get_cos_sim_scores                  data_model_helper.py:174-239
  get_final_second_attention_score    data_model_helper.py:416-443
  get_top_k_recommendations           (new) the k best news of the table (or of a pool of it) per user, scored like
                                      get_final_score when given the classification baseline

Same positional signatures and return types (CPU tensors / numpy) as the reference; the work is
one table upload + one dense row transform (cached per table/weights) + one fused CUDA launch
instead of a DataLoader, a per-impression Python loop and a per-impression scipy call.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from .data_utils import rank_group_preds, ranks_to_object_array
from .engine import cached_engine, host_base, host_pool


def get_final_attention_eval(history_rev_index: np.ndarray, history_len_list: np.ndarray,
                             news_embeddings: torch.Tensor, model: torch.nn.Module, precision=None) -> torch.Tensor:
    eng = cached_engine(news_embeddings, model, None, precision=precision)
    return eng.user_vectors(history_rev_index, history_len_list).cpu()


def get_cos_sim_scores(history_rev_index: np.ndarray, history_len_list: np.ndarray, news_rev_index: np.ndarray,
                       impression_len_list: np.ndarray, news_embeddings: torch.Tensor, model: torch.nn.Module,
                       query_news_embeddings: Optional[torch.Tensor] = None, precision=None) -> torch.Tensor:
    assert len(history_len_list) == len(impression_len_list), "Number of rows should be consistent"
    assert int(np.sum(impression_len_list)) == len(news_rev_index), \
        "Number of impressions should match length of impression list"
    q = query_news_embeddings if isinstance(query_news_embeddings, torch.Tensor) else None
    eng = cached_engine(news_embeddings, model, q, precision=precision)
    _, scores, _ = eng.score(history_rev_index, history_len_list, news_rev_index, impression_len_list,
                             want_ranks=False)
    return scores.cpu()


def get_final_second_attention_score(history_rev_index: np.ndarray, history_len_list: np.ndarray,
                                     news_rev_index: np.ndarray, impression_len_list: np.ndarray,
                                     news_embeddings: torch.Tensor, history_bool, attention_model: torch.nn.Module,
                                     precision=None) -> dict:
    """{"scores": float32[sum C], "grouped_scores": object[I] of dense-rank arrays}.

    Like the reference this expects `history_*` to describe exactly the impressions selected by
    `history_bool` (scripts/eval.py loads the WITH_HISTORY subset, so it is all True)."""
    hb = np.asarray(history_bool, dtype=bool)
    imp_len = np.asarray(impression_len_list)
    cand_idx = np.asarray(news_rev_index)[np.repeat(hb, imp_len)]
    cand_len = imp_len[hb]
    eng = cached_engine(news_embeddings, attention_model, None, precision=precision)
    _, scores, ranks = eng.score(history_rev_index, history_len_list, cand_idx, cand_len, want_ranks=True)
    scores_np = scores.cpu().numpy()
    if hb.all():
        grouped = ranks_to_object_array(ranks.cpu().numpy(), imp_len)
    else:
        # the reference ranks the filtered scores against the UNFILTERED length list
        # (data_model_helper.py:442); reproduce that grouping
        grouped = rank_group_preds(scores_np, imp_len)
    return {"scores": scores_np, "grouped_scores": grouped}


def get_top_k_recommendations(history_rev_index: np.ndarray, history_len_list: np.ndarray,
                              news_embeddings: torch.Tensor, model: torch.nn.Module, k: int = 10,
                              exclude_history: bool = True, query_news_embeddings: Optional[torch.Tensor] = None,
                              precision=None, pool=None, classification_score: Optional[np.ndarray] = None,
                              weight_model=None, history_bool=None) -> dict:
    """The k news that score best against each user (no counterpart in the reference, which only scores the candidate
    lists of the impressions).  Same user vector and cosine as `get_cos_sim_scores`; with `exclude_history` a user's
    own history is never recommended.

    `pool` (row ids, or a bool mask over the table) restricts the news to those rows, e.g. the news of an evaluation
    period's impressions.  With `classification_score` (one classification-head score per table row,
    `get_classification_preds`) the score is `get_final_score`'s: sigmoid(alpha) * cosine + (1 - sigmoid(alpha)) *
    classification score (alpha of `weight_model`; pure cosine without one), and the classification score alone for
    users without a history.  `history_bool` (as in `get_final_score`) marks the behaviour rows that have a history;
    `history_*` then describe those rows only, and the result has one list per behaviour row.

    Returns numpy {"top_k_rows": int32 [U, k] (row ids = `news_list` positions), "top_k_scores": float32 [U, k]},
    each list by score descending then row id ascending, -1 / NaN where a user has fewer than k eligible news.
    1 <= k <= 32."""
    n_rows = news_embeddings.shape[0]
    if history_bool is not None and classification_score is None:
        raise ValueError("history_bool needs classification_score: users without a history are recommended by the "
                         "classification baseline alone")
    base = None if classification_score is None else host_base(classification_score, n_rows)
    pool = None if pool is None else host_pool(pool, n_rows)
    hist_len = history_len_list if history_bool is None else _full_history_lengths(history_len_list, history_bool)
    alpha = weight_model.blend_alpha() if weight_model is not None else 1.0
    q = query_news_embeddings if isinstance(query_news_embeddings, torch.Tensor) else None
    eng = cached_engine(news_embeddings, model, q, precision=precision)
    rows, scores = eng.recommend(history_rev_index, hist_len, k, exclude_history=exclude_history, pool=pool,
                                 cand_base=base, blend_alpha=alpha)
    return {"top_k_rows": rows.cpu().numpy(), "top_k_scores": scores.cpu().numpy()}


def get_classification_preds(news_embeddings: torch.Tensor, model: torch.nn.Module) -> np.ndarray:
    """Classification-head score per table row (data_model_helper.py:91-98): float32 [N]."""
    from . import _lib

    dev = _lib.require_device()
    out = []
    with torch.cuda.device(dev):
        for r0 in range(0, news_embeddings.shape[0], 46336):  # the reference's batch size (:94)
            out.append(model(news_embeddings[r0:r0 + 46336].to(dev)).squeeze(dim=-1).float().cpu())
    return torch.cat(out).numpy()


def get_classification_baseline_scores(news_embeddings: torch.Tensor, model: torch.nn.Module,
                                       news_rev_index: np.ndarray) -> dict:
    preds = get_classification_preds(news_embeddings, model)
    return {"classification_preds": preds, "baseline_scores": preds[news_rev_index]}


def _full_history_lengths(history_len_list, history_bool) -> np.ndarray:
    """history_len_list only has entries for impressions WITH history (data_utils.py:183-185): expand to one
    length per impression (0 where history_bool is False)."""
    hb = np.asarray(history_bool, dtype=bool)
    full = np.zeros(hb.shape[0], dtype=np.int32)
    full[hb] = np.asarray(history_len_list, dtype=np.int32)
    return full


def get_final_score(history_rev_index: np.ndarray, history_len_list: np.ndarray, news_rev_index: np.ndarray,
                    impression_len_list: np.ndarray, news_embeddings: torch.Tensor, classification_score: np.ndarray,
                    history_bool, attention_model: torch.nn.Module, weight_model,
                    query_news_embeddings: Optional[torch.Tensor] = None, precision=None) -> dict:
    """data_model_helper.py:272-301: impressions with history get sigmoid(alpha)*cosine + (1-sigmoid(alpha))*
    classification score, the others the classification score alone; then dense ranks per impression.  One fused
    launch over ALL impressions (the blend and the no-history fallback live in `nrb_score_rank`)."""
    q = query_news_embeddings if isinstance(query_news_embeddings, torch.Tensor) else None
    eng = cached_engine(news_embeddings, attention_model, q, precision=precision)
    alpha = weight_model.blend_alpha() if weight_model is not None else 1.0
    hist_len_full = _full_history_lengths(history_len_list, history_bool)
    _, scores, ranks = eng.score(history_rev_index, hist_len_full, news_rev_index, impression_len_list,
                                 want_ranks=True, cand_base=np.asarray(classification_score, dtype=np.float32),
                                 blend_alpha=alpha)
    return {"scores": scores.cpu().numpy(),
            "grouped_scores": ranks_to_object_array(ranks.cpu().numpy(), np.asarray(impression_len_list))}


def get_final_only_attention_score(history_rev_index: np.ndarray, history_len_list: np.ndarray,
                                   news_rev_index: np.ndarray, impression_len_list: np.ndarray,
                                   news_embeddings: torch.Tensor, classification_score: np.ndarray, history_bool,
                                   attention_model: torch.nn.Module,
                                   query_news_embeddings: Optional[torch.Tensor] = None, precision=None) -> dict:
    """data_model_helper.py:304-335: pure cosine for impressions with history, classification score otherwise."""
    return get_final_score(history_rev_index, history_len_list, news_rev_index, impression_len_list, news_embeddings,
                           classification_score, history_bool, attention_model, None,
                           query_news_embeddings=query_news_embeddings, precision=precision)
