"""Drop-in pipeline components around the hot path (reference: news_rec_utils/components.py).

  TransformData              components.py:45-114   behaviour log -> row ids + CSR index arrays (native builder)
  SaveEmbeddingComponent     components.py:178-222  table writer  (`<dataset>.pt`, `query_<dataset>.pt`)
  LoadEmbeddingComponent     components.py:225-258  table reader
  FinalAttentionComponent    components.py:980-1027 gather + user encoder + cosine + dense rank
  TopKRecommendationComponent (new)                 the k best news of the table (or of the impressions) per user

Only `transform` is in scope (scripts/eval.py's path); training stays with the reference."""
from __future__ import annotations

from pathlib import Path
from typing import Any, Optional

import numpy as np
import torch

from .data_model_helper import get_classification_preds, get_final_second_attention_score, get_top_k_recommendations
from .data_utils import split_impressions_and_history
from .modeling_utils import get_final_attention_model
from .pipeline import PipelineComponent, check_req_keys


class TransformData(PipelineComponent):
    """Parses the behaviour log into the hot path's input layout and lines the per-news side tables up with the
    row ids (`news_list` order = first appearance).  Same keys in and out as the reference."""

    required_keys = {"behaviors", "news_text_dict", "news_category", "news_subcategory", "news_title_entity",
                     "news_abstract_entity"}
    _consumed = ("behaviors", "news_title_entity", "news_abstract_entity", "news_category", "news_subcategory")

    def transform(self, context_dict: dict[str, Any]) -> dict[str, Any]:
        check_req_keys(self.required_keys, context_dict)
        behaviors = context_dict["behaviors"]
        out = {k: v for k, v in context_dict.items() if k not in self._consumed}
        out["ImpressionID"] = behaviors["ImpressionID"]
        out.update(split_impressions_and_history(list(behaviors["Impressions"]), list(behaviors["History"])))
        out["history_bool"] = behaviors["History"].notna()
        rows = out["news_list"]
        per_row = lambda table, dtype: torch.from_numpy(np.asarray([table[n] for n in rows], dtype=dtype))
        out["title_entity_embed"] = per_row(context_dict["news_title_entity"], np.float32)
        out["abstract_entity_embed"] = per_row(context_dict["news_abstract_entity"], np.float32)
        out["cat_indices"] = per_row(context_dict["news_category"], np.int32).unsqueeze(dim=-1)
        out["subcat_indices"] = per_row(context_dict["news_subcategory"], np.int32).unsqueeze(dim=-1)
        return out


def _table_paths(save_dir: Path, dataset) -> tuple[Path, Path]:
    name = getattr(dataset, "value", dataset)  # NewsDataset member (or its plain name)
    return Path(save_dir) / f"{name}.pt", Path(save_dir) / f"query_{name}.pt"


class SaveEmbeddingComponent(PipelineComponent):
    """Writes the news-embedding table (and the query-side table when present) as CPU tensors."""

    required_keys = {"news_embeddings", "news_dataset"}

    def __init__(self, save_dir: Path):
        self.save_dir = Path(save_dir)

    def transform(self, context_dict: dict[str, Any]) -> dict[str, Any]:
        check_req_keys(self.required_keys, context_dict)
        self.save_dir.mkdir(parents=True, exist_ok=True)
        table_path, query_path = _table_paths(self.save_dir, context_dict["news_dataset"])
        torch.save(context_dict["news_embeddings"], table_path)
        if "query_news_embeddings" in context_dict:
            torch.save(context_dict["query_news_embeddings"], query_path)
        return context_dict


class LoadEmbeddingComponent(PipelineComponent):
    """Reads the table(s) back; the scoring engine uploads them once and keeps them resident (`cached_engine`)."""

    required_keys = {"news_dataset"}

    def __init__(self, save_dir: Path):
        self.save_dir = Path(save_dir)

    def transform(self, context_dict: dict[str, Any]) -> dict[str, Any]:
        check_req_keys(self.required_keys, context_dict)
        table_path, query_path = _table_paths(self.save_dir, context_dict["news_dataset"])
        context_dict["news_embeddings"] = torch.load(table_path, weights_only=True)
        if query_path.exists():
            context_dict["query_news_embeddings"] = torch.load(query_path, weights_only=True)
        return context_dict


class FinalAttentionComponent(PipelineComponent):
    required_keys = {
        "news_embeddings",
        "impression_rev_ind_array",
        "impression_len_list",
        "history_rev_ind_array",
        "history_len_list",
        "history_bool",
    }
    train_required_keys = required_keys | {"labels"}

    def __init__(self, attention_model_path: Optional[Path] = None, attention_model=None, precision=None, **_unused):
        self.attention_model = attention_model if attention_model is not None else \
            get_final_attention_model(attention_model_path)
        self.precision = precision

    def transform(self, context_dict: dict[str, Any]) -> dict[str, Any]:
        check_req_keys(self.required_keys, context_dict)
        out = context_dict.copy()
        out.update(get_final_second_attention_score(
            out["history_rev_ind_array"][0], out["history_len_list"], out["impression_rev_ind_array"][0],
            out["impression_len_list"], out["news_embeddings"], out["history_bool"], self.attention_model,
            precision=self.precision))
        return out

    def train(self, context_dict, val_context_dict=None) -> None:
        raise NotImplementedError("training is out of scope for the B200 hot path (use the reference trainer)")


class TopKRecommendationComponent(PipelineComponent):
    """Recommends, for every user with a history, the k news of the whole table that score best against the user
    vector (the cosine FinalAttentionComponent ranks candidates by), history excluded by default.  Adds
    `top_k_rows` (int32 [U, k] row ids), `top_k_scores` (float32 [U, k]) and `top_k_news` (object [U, k] news ids
    from `news_list`, None where a user has fewer than k eligible news).

    With `classification_model` the news are scored like `get_final_score`: the cosine blended with the model's
    per-news classification score (weight of `weight_model`), and users without a history get the classification
    score alone; the context then needs `history_bool` and there is one list per behaviour row.
    `restrict_to_impressions` draws the news from those that occur in `impression_rev_ind_array` only."""

    required_keys = {"news_embeddings", "history_rev_ind_array", "history_len_list", "news_list"}

    def __init__(self, k: int = 10, attention_model_path: Optional[Path] = None, attention_model=None,
                 exclude_history: bool = True, precision=None, classification_model=None, weight_model=None,
                 restrict_to_impressions: bool = False, **_unused):
        self.k = int(k)
        self.attention_model = attention_model if attention_model is not None else \
            get_final_attention_model(attention_model_path)
        self.exclude_history = exclude_history
        self.precision = precision
        self.classification_model = classification_model
        self.weight_model = weight_model
        self.restrict_to_impressions = restrict_to_impressions

    def transform(self, context_dict: dict[str, Any]) -> dict[str, Any]:
        req = set(self.required_keys)
        if self.classification_model is not None:
            req.add("history_bool")
        if self.restrict_to_impressions:
            req.add("impression_rev_ind_array")
        check_req_keys(req, context_dict)
        out = context_dict.copy()
        extra = {}
        if self.classification_model is not None:
            extra = {"classification_score": get_classification_preds(out["news_embeddings"], self.classification_model),
                     "weight_model": self.weight_model, "history_bool": out["history_bool"]}
        if self.restrict_to_impressions:
            extra["pool"] = np.unique(np.asarray(out["impression_rev_ind_array"][0]))
        res = get_top_k_recommendations(
            out["history_rev_ind_array"][0], out["history_len_list"], out["news_embeddings"], self.attention_model,
            k=self.k, exclude_history=self.exclude_history, query_news_embeddings=out.get("query_news_embeddings"),
            precision=self.precision, **extra)
        out.update(res)
        news = np.asarray(out["news_list"], dtype=object)
        rows = res["top_k_rows"]
        top = np.full(rows.shape, None, dtype=object)
        top[rows >= 0] = news[rows[rows >= 0]]
        out["top_k_news"] = top
        return out
