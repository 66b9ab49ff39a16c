"""Vectorised references of the one-warp-per-item kernels, computed over every group at once.

The per-group oracles (`oracle.rank_group_preds`, `oracle.score_row`, a stable numpy argsort per group) take seconds
to minutes on the hundreds of thousands of groups a test needs to give every warp of a grid-stride kernel several
items.  These functions restate the same definitions with one sort over all groups; `tests/test_segment_oracle_cpu.py`
holds them to the per-group oracles.
"""
from __future__ import annotations

import numpy as np
import torch


def csr(counts) -> np.ndarray:
    off = np.zeros(len(counts) + 1, dtype=np.int64)
    np.cumsum(counts, out=off[1:])
    return off


def dense_rank_segments(scores: torch.Tensor, offsets: torch.Tensor):
    """`rank_group_preds` of every group at once (any device, the scores' own dtype).

    Returns (ranks int32 [n]: descending dense ranks, equal values (-0.0 == 0.0) share a rank, 0 for every member of
    a group that holds a NaN; min_gap float64 [groups]: the smallest difference of two adjacent sorted scores of the
    group, 0 where two are equal, inf for groups of fewer than two, NaN for a group with a NaN)."""
    dev = scores.device
    n, n_groups = scores.numel(), offsets.numel() - 1
    grp = torch.repeat_interleave(torch.arange(n_groups, device=dev), offsets[1:] - offsets[:-1])
    order = torch.sort(scores, descending=True, stable=True).indices
    order = order[torch.sort(grp[order], stable=True).indices]  # by group, then score descending
    s, g = scores[order], grp[order]
    same = g[1:] == g[:-1]
    new = torch.ones(n, dtype=torch.int64, device=dev)
    new[1:] = (~same | (s[1:] != s[:-1])).long()
    c = torch.cumsum(new, 0)
    ranks = torch.empty(n, dtype=torch.int64, device=dev)
    ranks[order] = c - c[offsets[:-1][g]] + 1
    has_nan = torch.zeros(n_groups, dtype=torch.int64, device=dev).index_add_(0, grp, torch.isnan(scores).long()) > 0
    ranks[has_nan[grp]] = 0
    min_gap = torch.full((n_groups,), float("inf"), dtype=torch.float64, device=dev)
    min_gap.scatter_reduce_(0, g[1:][same], (s[:-1] - s[1:]).double()[same], "amin")
    min_gap[has_nan] = float("nan")
    return ranks.to(torch.int32), min_gap


def topk_order_segments(scores: np.ndarray, counts, ks) -> list:
    """`nrb_topk_order` for each k of `ks`: out[g, p] = position within group g of the candidate at place p of
    np.argsort(-scores, kind="stable") with NaN after every number (among themselves by position), -1 past the
    group's end."""
    counts = np.asarray(counts, dtype=np.int64)
    off = csr(counts)
    n = int(off[-1])
    grp = np.repeat(np.arange(len(counts)), counts)
    pos = np.arange(n) - off[grp]
    nan = np.isnan(scores)
    key = np.where(nan, 0.0, -np.asarray(scores, dtype=np.float64))
    order = np.lexsort((pos, key, nan, grp))  # last key first: group, NaN flag, -score, position
    g, place, who = grp[order], np.arange(n) - off[grp[order]], pos[order]
    outs = []
    for k in ks:
        out = np.full((len(counts), k), -1, dtype=np.int32)
        m = place < k
        out[g[m], place[m]] = who[m]
        outs.append(out)
    return outs


def mind_metrics_segments(ranks: np.ndarray, labels: np.ndarray, counts) -> np.ndarray:
    """`oracle.score_row` of every impression at once: float64 [I, 4] = AUC, MRR, nDCG@5, nDCG@10.

    y_score = 1 / rank, and the order is np.argsort(y_score, kind="stable")[::-1]: the higher score first and, among
    equal scores, the LATER candidate first (the tie order `nrb_mind_metrics` documents; the reference's own numpy
    default argsort is not stable).  The ideal order is the same over the labels.  Gains 2^y - 1, discounts
    log2(place + 2); AUC counts (positive, negative) pairs with equal scores 1/2.  NaN rows: empty impressions,
    a single class, or a rank 0 (NaN group)."""
    counts = np.asarray(counts, dtype=np.int64)
    n_imp = len(counts)
    off = csr(counts)
    n = int(off[-1])
    r = np.asarray(ranks, dtype=np.int64)
    y = np.asarray(labels, dtype=np.float64)
    grp = np.repeat(np.arange(n_imp), counts)
    pos = np.arange(n) - off[grp]
    with np.errstate(divide="ignore"):
        y_score = 1.0 / r.astype(np.float64)

    def places(key):
        o = np.lexsort((-pos, -key, grp))  # by group, key descending, later candidate first
        p = np.empty(n, dtype=np.int64)
        p[o] = np.arange(n) - off[grp[o]]
        return p

    place, iplace = places(y_score), places(y)
    sums = lambda v: np.bincount(grp, weights=v, minlength=n_imp)
    gain = 2.0 ** y - 1.0
    dcg = lambda p, k: sums(np.where(p < k, gain / np.log2(p + 2.0), 0.0))
    is_pos = y > 0.5
    n_pos, n_neg = sums(is_pos.astype(np.float64)), sums((~is_pos).astype(np.float64))
    # AUC numerator: for every positive, the negatives of its group with a lower score (a larger rank) + half the
    # negatives with the same rank
    span = int(r.max(initial=0)) + 2
    key = grp * span + r
    neg = np.sort(key[~is_pos])
    kp, gp = key[is_pos], grp[is_pos]
    lo, hi = np.searchsorted(neg, kp, "left"), np.searchsorted(neg, kp, "right")
    end = np.searchsorted(neg, gp * span + span, "left")
    auc_num = np.bincount(gp, weights=(end - hi) + 0.5 * (hi - lo), minlength=n_imp)
    bad = sums((r <= 0).astype(np.float64)) > 0
    valid = ~bad & (n_pos > 0) & (n_neg > 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        per = np.stack([auc_num / (n_pos * n_neg), sums(y / (place + 1.0)) / sums(y),
                        dcg(place, 5) / dcg(iplace, 5), dcg(place, 10) / dcg(iplace, 10)], axis=1)
    per[~valid] = np.nan
    return per


def pool_score_fp64(mode: int, X: torch.Tensor, E, T: torch.Tensor, hist_idx: torch.Tensor, hist_off: torch.Tensor,
                    cand_idx: torch.Tensor, cand_off: torch.Tensor, base=None, alpha: float = 1.0,
                    max_elems: int = 1 << 27):
    """fp64 user vectors [I, d] and scores [C] of `nrb_score_rank` on the same (already rounded) tables, on their
    device, in chunks of impressions whose gathered rows hold at most `max_elems` values.

    mode 0 (FinalAttention): u = sum(x * e) / (sum(e) + 1e-10); mode 1 (mean + L2): u = mean(x) / max(|mean|, 1e-12),
    an empty history giving 0 / 0 = NaN.  score = (u / max(|u|, 1e-8)) . (c / max(|c|, 1e-8)); with a baseline,
    alpha * score + (1 - alpha) * base[c], or base[c] alone for an impression without history."""
    dev = X.device
    X64, T64 = X.double(), T.double()
    E64 = E.double() if mode == 0 else None
    Tn = T64 / T64.norm(dim=1, keepdim=True).clamp_min(1e-8)
    b64 = base.double() if base is not None else None
    n_imp, d = hist_off.numel() - 1, X.shape[1]
    ho, co = hist_off.cpu().numpy(), cand_off.cpu().numpy()
    hlen, clen = hist_off[1:] - hist_off[:-1], cand_off[1:] - cand_off[:-1]
    user = torch.empty(n_imp, d, dtype=torch.float64, device=dev)
    scores = torch.empty(int(co[-1]), dtype=torch.float64, device=dev)
    rows = max(1, max_elems // d)
    i0 = 0
    while i0 < n_imp:
        i1 = min(np.searchsorted(ho, ho[i0] + rows, "right"), np.searchsorted(co, co[i0] + rows, "right")) - 1
        i1 = min(max(int(i1), i0 + 1), n_imp)
        n = i1 - i0
        h = hist_idx[ho[i0]:ho[i1]].long()
        owner = torch.repeat_interleave(torch.arange(n, device=dev), hlen[i0:i1])
        if mode == 0:
            e = E64[h]
            num = torch.zeros(n, d, dtype=torch.float64, device=dev).index_add_(0, owner, X64[h] * e)
            den = torch.zeros(n, d, dtype=torch.float64, device=dev).index_add_(0, owner, e)
            u = num / (den + 1e-10)
        else:
            u = torch.zeros(n, d, dtype=torch.float64, device=dev).index_add_(0, owner, X64[h])
            u = u / hlen[i0:i1, None].double()
            u = u / u.norm(dim=1, keepdim=True).clamp_min(1e-12)
        user[i0:i1] = u
        un = u / u.norm(dim=1, keepdim=True).clamp_min(1e-8)
        c = cand_idx[co[i0]:co[i1]].long()
        cown = torch.repeat_interleave(torch.arange(n, device=dev), clen[i0:i1])
        s = (un[cown] * Tn[c]).sum(1)
        if b64 is not None:
            s = torch.where((hlen[i0:i1] > 0)[cown], alpha * s + (1 - alpha) * b64[c], b64[c])
        scores[co[i0]:co[i1]] = s
        i0 = i1
    return user, scores
