"""Tensor-level wrappers over the C ABI (device tensors in, device tensors out).

These are the only places that call into libnrb200.so.  Every wrapper validates
device / dtype / contiguity, passes raw pointers + the current torch stream and
raises on a non-zero status.  No wrapper has a PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import BF16, F32, LatentWeights, check, dtype_code, load, ptr, require_device, stream_ptr


def _dev(t: torch.Tensor, name: str, dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.NrbError(f"{name} must be a CUDA tensor")
    if dtype is not None and t.dtype != dtype:
        raise _lib.NrbError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _lib.NrbError(f"{name} must be contiguous")
    return t


def new_err_flag(device) -> torch.Tensor:
    return torch.zeros(1, dtype=torch.int32, device=device)


def raise_on_index_error(flag: torch.Tensor, what: str) -> None:
    """Host-side check of the device error flag (synchronises)."""
    f = int(flag.item())
    if f & 1:
        raise IndexError(f"{what}: row index out of range for the embedding table")
    if f & 2:
        raise OverflowError(f"{what}: a dense rank does not fit int16 (ask for int32 ranks)")


def dense_rank(scores: torch.Tensor, offsets: torch.Tensor) -> torch.Tensor:
    """int32 dense ranks (0 = NaN group).  rank_group_preds, data_utils.py:414-415.
    float32 or float64 scores, ranked in their own dtype like scipy does."""
    require_device(scores.device)
    _dev(scores, "scores")
    if scores.dtype not in (torch.float32, torch.float64):
        raise _lib.NrbError(f"scores must be float32 or float64, got {scores.dtype}")
    _dev(offsets, "offsets", torch.int64)
    n_groups = offsets.numel() - 1
    ranks = torch.empty(scores.numel(), dtype=torch.int32, device=scores.device)
    fn = load().nrb_dense_rank if scores.dtype == torch.float32 else load().nrb_dense_rank_f64
    check(fn(ptr(scores), ptr(offsets), n_groups, ptr(ranks), stream_ptr()), "nrb_dense_rank")
    return ranks


def narrow_ranks(ranks: torch.Tensor, out: torch.Tensor, err_flag: torch.Tensor) -> torch.Tensor:
    """int32 dense ranks -> int16 (nrb_narrow_ranks); bit 1 of err_flag is set if a rank exceeds 32767."""
    require_device(ranks.device)
    _dev(ranks, "ranks", torch.int32)
    _dev(out, "out", torch.int16)
    if out.numel() != ranks.numel():
        raise _lib.NrbError("narrow_ranks: size mismatch")
    check(load().nrb_narrow_ranks(ptr(ranks), ptr(out), ranks.numel(), ptr(err_flag), stream_ptr()), "nrb_narrow_ranks")
    return out


def topk_order(scores: torch.Tensor, offsets: torch.Tensor, k: int) -> torch.Tensor:
    """int32 [n_groups, k]: positions of each group's k best candidates in descending score order (stable),
    -1 padded (nrb_topk_order)."""
    require_device(scores.device)
    _dev(scores, "scores", torch.float32)
    _dev(offsets, "offsets", torch.int64)
    n_groups = offsets.numel() - 1
    out = torch.empty(n_groups, k, dtype=torch.int32, device=scores.device)
    check(load().nrb_topk_order(ptr(scores), ptr(offsets), n_groups, int(k), ptr(out), stream_ptr()), "nrb_topk_order")
    return out


def gather_collate(table: torch.Tensor, idx: torch.Tensor, offsets: torch.Tensor, max_len: int,
                   err_flag: Optional[torch.Tensor] = None):
    """final_attention_eval_collate_fn on device (data_utils.py:784-791)."""
    dev = require_device(table.device)
    _dev(table, "table")
    _dev(idx, "idx", torch.int32)
    _dev(offsets, "offsets", torch.int64)
    n_groups = offsets.numel() - 1
    n_rows, dim = table.shape
    emb = torch.empty(n_groups, max_len, dim, dtype=table.dtype, device=dev)
    mask = torch.empty(n_groups, max_len, dtype=torch.int32, device=dev)
    flag = err_flag if err_flag is not None else new_err_flag(dev)
    check(load().nrb_gather_collate(ptr(table), dtype_code(table.dtype), n_rows, dim, table.stride(0), ptr(idx),
                                    ptr(offsets), n_groups, max_len, ptr(emb), ptr(mask), ptr(flag), stream_ptr()),
          "nrb_gather_collate")
    if err_flag is None:
        raise_on_index_error(flag, "gather_collate")
    return emb, mask


def mask_to_csr(mask: torch.Tensor):
    """attention_mask [B, S] (any dtype, 0 = padded) -> (idx int32 [B*S] of valid flat slots, off int64 [B+1]) on the
    device (nrb_mask_to_csr); no host synchronisation, entries of idx beyond off[B] are unspecified."""
    dev = require_device(mask.device)
    if mask.dim() != 2:
        raise _lib.NrbError("attention_mask must be [batch, seq]")
    m = mask if mask.dtype == torch.int32 and mask.is_contiguous() else (mask != 0).to(torch.int32).contiguous()
    B, S = m.shape
    idx = torch.empty(max(B * S, 1), dtype=torch.int32, device=dev)
    off = torch.empty(B + 1, dtype=torch.int64, device=dev)
    ws = torch.empty(2 * B + 2, dtype=torch.int32, device=dev)
    check(load().nrb_mask_to_csr(ptr(m), B, S, ptr(idx), ptr(off), ptr(ws), stream_ptr()), "nrb_mask_to_csr")
    return idx, off


def pool_masked_rows(x: torch.Tensor, e: torch.Tensor, attention_mask: torch.Tensor) -> torch.Tensor:
    """exp-weighted masked pooling of per-slot rows x, e [B*S, d] (FinalAttention / NewAttention forward,
    modeling_utils.py:224-228): fp32 [B, d]."""
    dev = x.device
    idx, off = mask_to_csr(attention_mask.to(dev))
    B = off.numel() - 1
    zeros = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    none_idx = torch.zeros(1, dtype=torch.int32, device=dev)
    user, _, _ = score_rank(_lib.POOL_FINAL_ATTENTION, x, e, x, idx, off, none_idx, zeros, 0, want_user=True,
                            want_ranks=False)
    return user


def pad_rows_for_kernel(t: torch.Tensor) -> torch.Tensor:
    """[rows, d] -> [rows, d rounded up to a 512-byte multiple], zero filled (native strided row copy)."""
    es = t.element_size()
    quantum = 512 // es
    rows, d = t.shape
    dpad = (d + quantum - 1) // quantum * quantum
    if dpad == d:
        return t
    out = torch.zeros(rows, dpad, dtype=t.dtype, device=t.device)
    if rows:
        convert_rows(t, t.dtype, out=out[:, :d])
    return out


def score_rank(pool_mode: int, hist_x: torch.Tensor, hist_e: Optional[torch.Tensor], cand: torch.Tensor,
               hist_idx: torch.Tensor, hist_off: torch.Tensor, cand_idx: torch.Tensor, cand_off: torch.Tensor,
               n_cand_total: int, want_user: bool = False, want_ranks: bool = True,
               err_flag: Optional[torch.Tensor] = None, out_scores: Optional[torch.Tensor] = None,
               out_ranks: Optional[torch.Tensor] = None, cand_base: Optional[torch.Tensor] = None,
               blend_alpha: float = 1.0):
    """Fused gather -> user vector -> cosine (-> blend with a per-row baseline) -> dense rank (nrb_score_rank).

    Row widths that are not a multiple of 512 bytes (e.g. 384 bf16 elements) run on zero-padded copies of the tables
    (`pad_rows_for_kernel`; the engine caches its own): zero columns change no pooled value, dot product or norm."""
    dev = require_device(hist_x.device)
    _dev(hist_x, "hist_x")
    if hist_x.dim() == 2 and (hist_x.shape[1] * hist_x.element_size()) % 512 != 0:
        d = hist_x.shape[1]
        px = pad_rows_for_kernel(hist_x)
        pc = px if cand is hist_x else pad_rows_for_kernel(_dev(cand, "cand", hist_x.dtype))
        pe = None if hist_e is None else pad_rows_for_kernel(_dev(hist_e, "hist_e", hist_x.dtype))
        user, scores, ranks = score_rank(pool_mode, px, pe, pc, hist_idx, hist_off, cand_idx, cand_off, n_cand_total,
                                         want_user=want_user, want_ranks=want_ranks, err_flag=err_flag,
                                         out_scores=out_scores, out_ranks=out_ranks, cand_base=cand_base,
                                         blend_alpha=blend_alpha)
        return (None if user is None else user[:, :d].contiguous()), scores, ranks
    _dev(cand, "cand", hist_x.dtype)
    if hist_e is not None:
        _dev(hist_e, "hist_e", hist_x.dtype)
        if hist_e.stride(0) != hist_x.stride(0):
            raise _lib.NrbError("hist_x and hist_e must share the row stride")
    for t, n in ((hist_idx, "hist_idx"), (cand_idx, "cand_idx")):
        _dev(t, n, torch.int32)
    for t, n in ((hist_off, "hist_off"), (cand_off, "cand_off")):
        _dev(t, n, torch.int64)
    n_imp = hist_off.numel() - 1
    if cand_off.numel() - 1 != n_imp:
        raise AssertionError("Number of rows should be consistent")  # data_model_helper.py:183-185
    n_rows, dim = cand.shape
    user = torch.empty(n_imp, dim, dtype=torch.float32, device=dev) if want_user else None
    scores = out_scores if out_scores is not None else torch.empty(max(n_cand_total, 1), dtype=torch.float32, device=dev)
    ranks = None
    if want_ranks:
        ranks = out_ranks if out_ranks is not None else torch.empty(max(n_cand_total, 1), dtype=torch.int32, device=dev)
    if cand_base is not None:
        _dev(cand_base, "cand_base", torch.float32)
        if cand_base.numel() < n_rows:
            raise _lib.NrbError("cand_base must have one entry per table row")
    flag = err_flag if err_flag is not None else new_err_flag(dev)
    check(load().nrb_score_rank(pool_mode, dtype_code(hist_x.dtype), dim, min(n_rows, hist_x.shape[0]),
                                ptr(hist_x), ptr(hist_e), hist_x.stride(0), ptr(cand), cand.stride(0),
                                ptr(cand_base), float(blend_alpha), ptr(hist_idx), ptr(hist_off), ptr(cand_idx), ptr(cand_off), n_imp,
                                ptr(user), ptr(scores), ptr(ranks), ptr(flag), stream_ptr()), "nrb_score_rank")
    if err_flag is None:
        raise_on_index_error(flag, "score_rank")
    if out_scores is None:
        scores = scores[:n_cand_total]
    if want_ranks and out_ranks is None:
        ranks = ranks[:n_cand_total]
    return user, scores, ranks


def _recommend_args(dim: int, k: int) -> None:
    """The limits of nrb_recommend, checked before anything touches a device."""
    if not 1 <= int(k) <= _lib.RECOMMEND_MAX_K:
        raise _lib.NrbError(f"recommend: k must be in [1, {_lib.RECOMMEND_MAX_K}] (got {k})")
    if dim <= 0 or dim % 64:
        raise _lib.NrbError(f"recommend: the embedding width must be a multiple of 64 (got {dim})")


def _recommend_pool_args(n_rows: int, n_users: int, pool, cand_base, hist_off) -> None:
    """dtype and shape checks of the pool / baseline / history arguments of `recommend`, before any device work."""
    if pool is not None:
        if not isinstance(pool, torch.Tensor) or pool.dtype != torch.int32 or pool.dim() != 1:
            raise _lib.NrbError("recommend: pool must be a 1-D int32 tensor of table row ids")
        if pool.numel() > n_rows:
            raise _lib.NrbError(f"recommend: a pool of distinct row ids has at most {n_rows} entries")
    if cand_base is not None:
        if not isinstance(cand_base, torch.Tensor) or cand_base.dtype != torch.float32 or cand_base.dim() != 1:
            raise _lib.NrbError("recommend: cand_base must be a 1-D float32 tensor")
        if cand_base.numel() != n_rows:
            raise _lib.NrbError(f"recommend: cand_base must have one entry per table row ({n_rows})")
    if hist_off is not None:
        if not isinstance(hist_off, torch.Tensor) or hist_off.dtype != torch.int64 or hist_off.dim() != 1:
            raise _lib.NrbError("recommend: hist_off must be a 1-D int64 tensor")
        if hist_off.numel() != n_users + 1:
            raise _lib.NrbError("recommend: hist_off must have U + 1 entries")


def recommend(table: torch.Tensor, users: torch.Tensor, k: int, table_op: Optional[torch.Tensor] = None,
              excl_idx: Optional[torch.Tensor] = None, excl_off: Optional[torch.Tensor] = None,
              err_flag: Optional[torch.Tensor] = None, pool: Optional[torch.Tensor] = None,
              cand_base: Optional[torch.Tensor] = None, blend_alpha: float = 1.0,
              hist_off: Optional[torch.Tensor] = None):
    """The k best rows of the table for each user (nrb_recommend_pool_blend): (rows int32 [U, k], scores fp32 [U, k]).

    score = cosine(user, row), ordered by score descending then row id ascending, (-1, NaN) once a user has no
    eligible rows left.  bf16 tables run the tensor-core GEMM on bf16 operands; fp32 tables run it on split-bf16
    operands (`table_op` = split_rows(table, 1), built here if not given).  The fp32 FFMA GEMM has no top-k epilogue,
    so fp32 retrieval always uses the split tensor-core path.  `excl_idx` / `excl_off` (int32 ids, int64 offsets
    [U + 1]): rows never returned for each user; an out-of-range id raises IndexError (or sets bit 0 of `err_flag`).

    `pool` (device int32 row ids, strictly ascending): only these rows are eligible and the GEMM runs over them alone;
    returned ids stay table row ids.  Ids out of range or not ascending raise IndexError like `excl_idx`.
    `cand_base` (device fp32 [N]) + `blend_alpha`: score = cos * alpha + base * (1 - alpha), or base alone for users
    whose history is empty in `hist_off` (device int64 [U + 1]; None: every user has a history) -- the blend and the
    fallback of `score_rank`.  NaN scores are never returned."""
    _recommend_args(table.shape[1] if table.dim() == 2 else 0, k)
    if users.dim() != 2:
        raise _lib.NrbError("users must be [U, d]")
    _recommend_pool_args(table.shape[0] if table.dim() == 2 else 0, users.shape[0], pool, cand_base, hist_off)
    dev = require_device(table.device)
    _dev(table, "table")
    _dev(users, "users", torch.float32)
    n_rows, dim = table.shape
    if users.shape[1] != dim:
        raise _lib.NrbError(f"users must be [U, {dim}]")
    prec = dtype_code(table.dtype)
    if table_op is None:
        table_op = table if prec == BF16 else split_rows(table, 1)
    _dev(table_op, "table_op", torch.bfloat16)
    if (excl_idx is None) != (excl_off is None):
        raise _lib.NrbError("excl_idx and excl_off go together")
    n_excl = 0
    if excl_idx is not None:
        _dev(excl_idx, "excl_idx", torch.int32)
        _dev(excl_off, "excl_off", torch.int64)
        if excl_off.numel() != users.shape[0] + 1:
            raise _lib.NrbError("excl_off must have U + 1 entries")
        n_excl = excl_idx.numel()
        if n_excl == 0:  # an empty id tensor may have no storage (NULL): nothing is excluded
            excl_idx = excl_off = None
    for t, n in ((pool, "pool"), (cand_base, "cand_base"), (hist_off, "hist_off")):
        if t is not None:
            _dev(t, n)
    n_pool = -1 if pool is None else pool.numel()
    U = users.shape[0]
    rows = torch.empty(U, k, dtype=torch.int32, device=dev)
    scores = torch.empty(U, k, dtype=torch.float32, device=dev)
    if U == 0:
        return rows, scores
    lib = load()
    ws_bytes = lib.nrb_recommend_pool_blend_workspace_bytes(prec, dim, n_rows, U, n_excl, int(k), n_pool)
    if ws_bytes == 0:
        check(-1, "nrb_recommend_pool_blend_workspace_bytes")
    ws = _workspace(dev, ws_bytes, "recommend")
    flag = err_flag if err_flag is not None else new_err_flag(dev)
    check(lib.nrb_recommend_pool_blend(prec, dim, n_rows, ptr(table), table.stride(0), ptr(table_op),
                                       table_op.stride(0), ptr(users), users.stride(0), U, ptr(excl_idx),
                                       ptr(excl_off), n_excl, int(k), ptr(pool), n_pool, ptr(cand_base),
                                       float(blend_alpha), ptr(hist_off), ptr(rows), ptr(scores), ptr(flag), ptr(ws),
                                       ws.numel(), stream_ptr()), "nrb_recommend_pool_blend")
    if err_flag is None:
        raise_on_index_error(flag, "recommend")
    return rows, scores


def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, epilogue: int = _lib.EPI_NONE,
           res: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None, group: int = 0,
           group_valid: int = 0) -> torch.Tensor:
    """y = epilogue(a @ w.T + bias).  bf16 operands -> tcgen05, fp32 operands -> FFMA."""
    dev = require_device(a.device)
    _dev(a, "a")
    _dev(w, "w", a.dtype)
    M, K = a.shape
    N = w.shape[0]
    if w.shape[1] != K:
        raise _lib.NrbError("a / w inner dimensions differ")
    out_dtype = out_dtype or a.dtype
    n_out = N // 2 if epilogue == _lib.EPI_GEGLU else N
    y = torch.empty(M, n_out, dtype=out_dtype, device=dev)
    if bias is not None:
        _dev(bias, "bias", torch.float32)
    if res is not None:
        _dev(res, "res", torch.float32)
    check(load().nrb_linear(dtype_code(a.dtype), epilogue, dtype_code(out_dtype), ptr(a), a.stride(0), ptr(w),
                            w.stride(0), ptr(bias), ptr(res), res.stride(0) if res is not None else 0, ptr(y),
                            y.stride(0), M, N, K, group, group_valid, stream_ptr()), "nrb_linear")
    return y


def final_attention_rows(table: torch.Tensor, weights: dict, out_dtype: torch.dtype,
                         x_out: Optional[torch.Tensor] = None, e_out: Optional[torch.Tensor] = None):
    """Per-row FinalAttention transform: (x, exp(logit)) tables (nrb_final_attention_rows).

    `weights`: linear{1..5}.weight in table.dtype, linear{1..4}.bias in fp32, on device.
    `x_out` / `e_out`: optional preallocated [n_rows, dim] row slices to write into."""
    dev = require_device(table.device)
    _dev(table, "table")
    n_rows, dim = table.shape
    hidden = weights["linear1.weight"].shape[0]
    prec = dtype_code(table.dtype)
    for i in range(1, 6):
        _dev(weights[f"linear{i}.weight"], f"linear{i}.weight", table.dtype)
    for i in range(1, 5):
        _dev(weights[f"linear{i}.bias"], f"linear{i}.bias", torch.float32)
    lib = load()
    ws_bytes = lib.nrb_final_attention_rows_workspace_bytes(prec, n_rows, dim, hidden)
    ws = _workspace(dev, ws_bytes, "fa")
    x = x_out if x_out is not None else torch.empty(n_rows, dim, dtype=out_dtype, device=dev)
    e = e_out if e_out is not None else torch.empty(n_rows, dim, dtype=out_dtype, device=dev)
    for t, nm in ((x, "x_out"), (e, "e_out")):
        _dev(t, nm, out_dtype)
        if tuple(t.shape) != (n_rows, dim):
            raise _lib.NrbError(f"{nm} must have shape {(n_rows, dim)}")
    check(lib.nrb_final_attention_rows(
        prec, dtype_code(out_dtype), ptr(table), table.stride(0), n_rows, dim, hidden,
        ptr(weights["linear1.weight"]), ptr(weights["linear1.bias"]),
        ptr(weights["linear2.weight"]), ptr(weights["linear2.bias"]),
        ptr(weights["linear3.weight"]), ptr(weights["linear3.bias"]),
        ptr(weights["linear4.weight"]), ptr(weights["linear4.bias"]),
        ptr(weights["linear5.weight"]), ptr(x), ptr(e), x.stride(0), ptr(ws), ws.numel(), stream_ptr()),
        "nrb_final_attention_rows")
    return x, e


def split_rows(src: torch.Tensor, role: int) -> torch.Tensor:
    """fp32 [rows, K] -> bf16 [rows, 3K]: [hi|hi|lo] (role 0, activations) or [hi|lo|hi] (role 1, weights)."""
    dev = require_device(src.device)
    _dev(src, "src", torch.float32)
    rows, K = src.shape
    out = torch.empty(rows, 3 * K, dtype=torch.bfloat16, device=dev)
    check(load().nrb_split_rows(ptr(src), src.stride(0), ptr(out), out.stride(0), rows, K, int(role), stream_ptr()),
          "nrb_split_rows")
    return out


def final_attention_rows_split(table: torch.Tensor, weights: dict, x_out: Optional[torch.Tensor] = None,
                               e_out: Optional[torch.Tensor] = None):
    """Per-row FinalAttention transform on the tensor cores at (almost) fp32 accuracy: fp32 table, weights
    `linear{1..5}.weight` pre-split by `split_rows(w, 1)`, fp32 biases -> fp32 (x, exp(logit)) tables."""
    dev = require_device(table.device)
    _dev(table, "table", torch.float32)
    n_rows, dim = table.shape
    hidden = weights["linear1.bias"].shape[0]
    for i in range(1, 6):
        _dev(weights[f"linear{i}.weight"], f"linear{i}.weight", torch.bfloat16)
    lib = load()
    ws_bytes = lib.nrb_final_attention_rows_split_workspace_bytes(n_rows, dim, hidden)
    ws = _workspace(dev, ws_bytes, "fa_split")
    x = x_out if x_out is not None else torch.empty(n_rows, dim, dtype=torch.float32, device=dev)
    e = e_out if e_out is not None else torch.empty(n_rows, dim, dtype=torch.float32, device=dev)
    check(lib.nrb_final_attention_rows_split(
        ptr(table), table.stride(0), n_rows, dim, hidden,
        ptr(weights["linear1.weight"]), ptr(weights["linear1.bias"]),
        ptr(weights["linear2.weight"]), ptr(weights["linear2.bias"]),
        ptr(weights["linear3.weight"]), ptr(weights["linear3.bias"]),
        ptr(weights["linear4.weight"]), ptr(weights["linear4.bias"]),
        ptr(weights["linear5.weight"]), ptr(x), ptr(e), x.stride(0), ptr(ws), ws.numel(), stream_ptr()),
        "nrb_final_attention_rows_split")
    return x, e


@dataclass
class FoldedLatent:
    """Device-resident, kernel-ready weights of one LatentAttentionModel."""

    precision: int
    dim: int
    heads: int
    dim_head: int
    num_latents: int
    latents_padded: int
    tensors: dict  # keeps the device tensors alive
    struct: LatentWeights


def latent_fold(sd: dict, heads: int, dim_head: int, precision: torch.dtype, device) -> FoldedLatent:
    """One-time weight preparation (nrb_latent_fold + GEGLU row interleave)."""
    L, dim = sd["latents"].shape
    Lp = max(32, 1 << (L - 1).bit_length())  # power of two: softmax groups tile the 256-column MMA tiles
    if precision == torch.bfloat16 and heads * Lp % 64:
        # the value GEMM contracts over heads * Lp, and the tensor-core GEMM takes K in multiples of 64
        raise _lib.NrbError(f"bf16 latent attention needs heads * latents_padded to be a multiple of 64 "
                            f"(got {heads} x {Lp}); use an even head count, more than 32 latents or fp32")
    dev = require_device(device)
    f32 = lambda k: sd[k].detach().to(device=dev, dtype=torch.float32).contiguous()
    lat = f32("latents")
    p0, p1 = "cross_attend_blocks.0.", "cross_attend_blocks.1."
    wq, wkv, wout = f32(p0 + "fn.to_q.weight"), f32(p0 + "fn.to_kv.weight"), f32(p0 + "fn.to_out.weight")
    if wq.shape != (heads * dim_head, dim):
        raise _lib.NrbError(f"to_q.weight has shape {tuple(wq.shape)}, expected {(heads * dim_head, dim)}")
    lnc_w, lnc_b = f32(p0 + "norm_context.weight"), f32(p0 + "norm_context.bias")
    prec = dtype_code(precision)
    lib = load()
    a = torch.empty(heads * Lp, dim, dtype=precision, device=dev)
    b = torch.empty(dim, heads * Lp, dtype=precision, device=dev)
    ws_bytes = lib.nrb_latent_fold_workspace_bytes(dim, heads, dim_head, L)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(lib.nrb_latent_fold(prec, dim, heads, dim_head, L, ptr(lat), ptr(lnc_w), ptr(lnc_b), ptr(wq), ptr(wkv),
                              ptr(wout), ptr(a), ptr(b), ptr(ws), ws_bytes, stream_ptr()), "nrb_latent_fold")
    # GEGLU: interleave the value / gate halves of net.0 in PAIRS (a0,a1,g0,g1,a2,a3,g2,g3,...) so that one
    # accumulator tile holds both and neighbouring columns form packed fp32 pairs (FFMA2 epilogue)
    w1, b1 = f32(p1 + "fn.net.0.weight"), f32(p1 + "fn.net.0.bias")
    half = w1.shape[0] // 2
    if half % 2:
        raise _lib.NrbError("GEGLU width must be even")
    w1i = torch.stack([w1[:half].view(half // 2, 2, dim), w1[half:].view(half // 2, 2, dim)], dim=1) \
        .reshape(2 * half, dim).to(precision).contiguous()
    b1i = torch.stack([b1[:half].view(half // 2, 2), b1[half:].view(half // 2, 2)], dim=1).reshape(2 * half).contiguous()
    t = {
        "a": a, "b": b,
        "ln1_w": f32(p0 + "norm.weight"), "ln1_b": f32(p0 + "norm.bias"),
        "ln2_w": f32(p1 + "norm.weight"), "ln2_b": f32(p1 + "norm.bias"),
        "w_ff1": w1i, "b_ff1": b1i,
        "w_ff2": f32(p1 + "fn.net.2.weight").to(precision).contiguous(), "b_ff2": f32(p1 + "fn.net.2.bias"),
    }
    torch.cuda.current_stream().synchronize()  # `ws` and the fp32 staging copies die here
    st = LatentWeights(prec, dim, heads, L, Lp, *(ptr(t[k]) for k in
                                                 ("a", "b", "ln1_w", "ln1_b", "ln2_w", "ln2_b", "w_ff1", "b_ff1",
                                                  "w_ff2", "b_ff2")))
    return FoldedLatent(prec, dim, heads, dim_head, L, Lp, t, st)


_ws_cache: dict = {}


def _workspace(dev: torch.device, nbytes: int, tag: str = "latent") -> torch.Tensor:
    """Grow-only scratch buffer per (device, tag, stream): avoids cudaMalloc in the steady state.  Keyed by
    the CURRENT stream as well, so that calls issued on different streams never share scratch memory (and a
    buffer that is replaced when it grows was only ever used on the stream the allocator frees it on)."""
    key = (dev.index, tag, torch.cuda.current_stream(dev).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = None
        _ws_cache.pop(key, None)
        buf = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _ws_cache[key] = buf
    return buf


def latent_forward(fw: FoldedLatent, x: torch.Tensor, mask: Optional[torch.Tensor], max_tokens: int = 65536):
    """LatentAttentionModel.forward on device: pooled [B,d] fp32 (mask given) or un-pooled [B,S,d]."""
    dev = require_device(x.device)
    _dev(x, "embeddings")
    B, S, d = x.shape
    if d != fw.dim:
        raise _lib.NrbError(f"embedding dim {d} != model dim {fw.dim}")
    lib = load()
    max_tokens = max(min(int(max_tokens), B * S), S)  # no larger than this call needs
    ws_bytes = lib.nrb_latent_forward_workspace_bytes(C.byref(fw.struct), max_tokens)
    ws = _workspace(dev, ws_bytes)
    if mask is not None:
        _dev(mask, "attention_mask", torch.int32)
        out = torch.empty(B, d, dtype=torch.float32, device=dev)
        pooled, unpooled = ptr(out), None
    else:
        out = torch.empty(B, S, d, dtype=torch.float32, device=dev)
        pooled, unpooled = None, ptr(out)
    ntok = C.c_int64(-1)
    check(lib.nrb_latent_forward(C.byref(fw.struct), ptr(x), dtype_code(x.dtype), B, S, ptr(mask), pooled, unpooled,
                                 ptr(ws), ws.numel(), max_tokens, C.byref(ntok), stream_ptr()), "nrb_latent_forward")
    return out


def mind_metrics(ranks: torch.Tensor, labels: torch.Tensor, offsets: torch.Tensor, want_per_impression: bool = True):
    """Per-impression AUC / MRR / nDCG@5 / nDCG@10 on device (nrb_mind_metrics).

    ranks int32 (dense, 0 = NaN group), labels int8, offsets int64 [I+1].
    Returns (per_imp float64 [I,4] | None, sums float64 [5] = metric sums + number of valid impressions)."""
    dev = require_device(ranks.device)
    _dev(ranks, "ranks", torch.int32)
    _dev(labels, "labels", torch.int8)
    _dev(offsets, "offsets", torch.int64)
    n_imp = offsets.numel() - 1
    per = torch.empty(n_imp, 4, dtype=torch.float64, device=dev) if want_per_impression else None
    sums = torch.zeros(5, dtype=torch.float64, device=dev)
    check(load().nrb_mind_metrics(ptr(ranks), ptr(labels), ptr(offsets), n_imp, ptr(per), ptr(sums), stream_ptr()),
          "nrb_mind_metrics")
    return per, sums


def push_rows(src: torch.Tensor, dst_ptrs: list, dst_dtype: torch.dtype, dst_row_offset: int, dst_stride: int) -> None:
    """All-gather building block: write the rows of `src` into every peer's full table (nrb_push_rows)."""
    require_device(src.device)
    _dev(src, "src")
    n_rows, dim = src.shape
    arr = (C.c_void_p * len(dst_ptrs))(*[int(p) for p in dst_ptrs])
    check(load().nrb_push_rows(ptr(src), dtype_code(src.dtype), src.stride(0), n_rows, dim, arr, len(dst_ptrs),
                               dtype_code(dst_dtype), dst_row_offset, dst_stride, stream_ptr()), "nrb_push_rows")


def push_bytes(src: torch.Tensor, dst_ptrs: list, dst_byte_offset: int) -> None:
    """Copy-engine all-gather step: the contiguous tensor `src` goes to every dst_ptrs[g] + offset (nrb_push_bytes)."""
    require_device(src.device)
    _dev(src, "src")
    arr = (C.c_void_p * len(dst_ptrs))(*[int(p) for p in dst_ptrs])
    check(load().nrb_push_bytes(ptr(src), src.numel() * src.element_size(), arr, len(dst_ptrs), dst_byte_offset,
                                stream_ptr()), "nrb_push_bytes")


def convert_rows(src: torch.Tensor, out_dtype: torch.dtype, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[rows, dim] fp32 <-> bf16 on the device (nrb_convert_rows): the table's way into HBM, no ATen copy kernel."""
    dev = require_device(src.device)
    if not src.is_cuda or src.dim() != 2 or src.stride(1) != 1:
        raise _lib.NrbError("src must be a CUDA [rows, dim] tensor with unit inner stride")
    rows, dim = src.shape
    if out is None:
        out = torch.empty(rows, dim, dtype=out_dtype, device=dev)
    if out.dtype != out_dtype or tuple(out.shape) != (rows, dim) or out.stride(1) != 1 or not out.is_cuda:
        raise _lib.NrbError("out must be a CUDA [rows, dim] tensor of the requested dtype")
    check(load().nrb_convert_rows(ptr(src), dtype_code(src.dtype), src.stride(0), ptr(out), dtype_code(out_dtype),
                                  out.stride(0), rows, dim, stream_ptr()), "nrb_convert_rows")
    return out


def push_attach(segments: list, spread: int) -> None:
    """Attach all-gather segments to the next `spread` tensor-core GEMM launches (nrb_push_attach).
    `segments`: [(src [rows, dim] CUDA tensor, multicast_ptr of the destination table, dst dtype, first dst row,
    dst row stride in elements)]; the GEMMs' spare warps multicast the rows to every rank (NVLS)."""
    arr = (_lib.PushSeg * max(len(segments), 1))()
    for i, (src, mc_ptr, dst_dtype, row0, dst_stride) in enumerate(segments):
        require_device(src.device)
        if src.dim() != 2 or src.stride(1) != 1:
            raise _lib.NrbError("push segment source must be a [rows, dim] tensor with unit inner stride")
        arr[i] = _lib.PushSeg(ptr(src), dtype_code(src.dtype), src.stride(0), int(mc_ptr), dtype_code(dst_dtype),
                              int(dst_stride), int(row0), src.shape[0], src.shape[1])
    check(load().nrb_push_attach(arr, len(segments), int(spread)), "nrb_push_attach")


def push_cancel() -> None:
    """Drop pending all-gather segments without sending them (error paths)."""
    load().nrb_push_cancel()


def push_flush() -> None:
    """Send what no GEMM picked up with the store-only multicast kernel (nrb_push_flush)."""
    check(load().nrb_push_flush(stream_ptr()), "nrb_push_flush")


def layer_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float,
               out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """Row-wise LayerNorm (nrb_layer_norm): x [rows, dim] fp32/bf16, gamma/beta fp32."""
    dev = require_device(x.device)
    _dev(x, "x")
    _dev(gamma, "gamma", torch.float32)
    _dev(beta, "beta", torch.float32)
    rows, dim = x.shape
    out_dtype = out_dtype or x.dtype
    y = torch.empty(rows, dim, dtype=out_dtype, device=dev)
    check(load().nrb_layer_norm(ptr(x), dtype_code(x.dtype), x.stride(0), ptr(gamma), ptr(beta), float(eps), ptr(y),
                                dtype_code(out_dtype), y.stride(0), rows, dim, stream_ptr()), "nrb_layer_norm")
    return y


_aux_streams: dict = {}


def _aux_stream(dev: torch.device) -> "torch.cuda.Stream":
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _aux_streams:
        _aux_streams[key] = torch.cuda.Stream(dev)
    return _aux_streams[key]


def latent_forward_packed(fw: FoldedLatent, tokens: torch.Tensor, item_off: torch.Tensor, max_tokens: int = 65536):
    """Varlen latent-attention pooling: tokens [T, d] (packed, fp32/bf16), item_off int64/int32 [B+1] on the
    host or device -> pooled [B, d] fp32.  Items are processed in chunks of at most `max_tokens` tokens."""
    dev = require_device(tokens.device)
    _dev(tokens, "tokens")
    T, d = tokens.shape
    if d != fw.dim:
        raise _lib.NrbError(f"token dim {d} != model dim {fw.dim}")
    off_host = item_off.detach().cpu().to(torch.int64)
    B = off_host.numel() - 1
    if int(off_host[-1]) != T or int(off_host[0]) != 0:
        raise _lib.NrbError("item_off must start at 0 and end at the number of tokens")
    lib = load()
    max_tokens = max(min(int(max_tokens), max(T, 1)), int((off_host[1:] - off_host[:-1]).max()) if B else 1)
    ws_bytes = lib.nrb_latent_forward_workspace_bytes(C.byref(fw.struct), max_tokens)
    ws = _workspace(dev, ws_bytes)
    out = torch.empty(B, d, dtype=torch.float32, device=dev)
    i0 = 0
    while i0 < B:
        # largest item range [i0, i1) whose tokens fit the workspace
        i1 = int(torch.searchsorted(off_host, off_host[i0] + max_tokens, right=True).item()) - 1
        i1 = max(i1, i0 + 1)
        t0, t1 = int(off_host[i0]), int(off_host[i1])
        # the few KB of offsets cross on a side stream: a pageable copy on the compute stream would make the host wait
        # for everything queued there (the previous chunk's pooling) and stall the caller's upload pipeline
        side = _aux_stream(dev)
        with torch.cuda.stream(side):
            local_off = (off_host[i0:i1 + 1] - t0).to(torch.int32).to(dev)
        torch.cuda.current_stream().wait_stream(side)
        local_off.record_stream(torch.cuda.current_stream())
        check(lib.nrb_latent_forward_packed(C.byref(fw.struct), ptr(tokens[t0:t1]), dtype_code(tokens.dtype), t1 - t0,
                                            ptr(local_off), i1 - i0, ptr(out[i0:i1]), ptr(ws), ws.numel(),
                                            stream_ptr()), "nrb_latent_forward_packed")
        i0 = i1
    return out
