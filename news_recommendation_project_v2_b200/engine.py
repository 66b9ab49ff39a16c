"""Device-resident scoring engine: table(s) + user-encoder row transform + fused score/rank.

This is the host-side owner of what the reference spreads over
`get_final_attention_eval` (data_model_helper.py:112-131, CPU gather in DataLoader
workers + per-batch H2D/D2H), the per-impression cosine loop (:200-230) and
`rank_group_preds` (data_utils.py:414-415).  Layout in HBM:

  cand table  T  [N, d]  row r = news_list[r]   (scored against; `news_embeddings`)
  hist tables X,E [N, d] FinalAttention's separable per-row outputs x and exp(logit)
                         (or a single transformed table for mean-pool encoders)
  CSR indices     int32 row ids + int64 offsets (from `*_rev_ind_array[0]` / `*_len_list`)

All arithmetic happens in libnrb200.so; torch only owns the buffers.
"""
from __future__ import annotations

import weakref
from typing import Optional

import numpy as np
import torch

from . import _lib, ops
from .config import LATENT_MAX_TOKENS, precision_dtype, precision_is_split
from .synthetic import csr_offsets

_table_cache: "dict[tuple, tuple[weakref.ref, torch.Tensor]]" = {}


def resident_table(table: torch.Tensor, dtype: torch.dtype, device: torch.device) -> torch.Tensor:
    """Upload (once) and cache a host table on the device in `dtype`."""
    if table.is_cuda and table.dtype == dtype and table.is_contiguous():
        return table
    key = (id(table), table.data_ptr(), tuple(table.shape), table.dtype, dtype, device.index, table._version)
    hit = _table_cache.get(key)
    if hit is not None and hit[0]() is table:
        return hit[1]
    # copy in the source dtype first (a pinned table then crosses PCIe by DMA) and convert on the GPU
    dev_t = table.detach().to(device=device, non_blocking=True).contiguous()
    if dev_t.dtype != dtype:
        if dev_t.dtype in (torch.float32, torch.bfloat16) and dev_t.dim() == 2:
            with torch.cuda.device(device):
                dev_t = ops.convert_rows(dev_t, dtype)  # native rounding kernel, not an ATen copy
        else:
            dev_t = dev_t.to(dtype)
    if len(_table_cache) > 8:
        _table_cache.clear()
    try:
        _table_cache[key] = (weakref.ref(table), dev_t)
    except TypeError:
        pass
    return dev_t


def _as_i32(a, device) -> torch.Tensor:
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=torch.int32).contiguous()
    arr = np.ascontiguousarray(np.asarray(a), dtype=np.int32)
    return torch.from_numpy(arr).to(device)


def _offsets(lengths, device) -> tuple[torch.Tensor, int]:
    if isinstance(lengths, torch.Tensor):
        lengths = lengths.detach().cpu().numpy()
    off = csr_offsets(np.asarray(lengths))
    return torch.from_numpy(off).to(device), int(off[-1])


def _final_attention_weights_split(model, device) -> dict:
    """fp32 weights -> [hi|lo|hi] bf16 operands of the split-bf16 tensor-core GEMMs (nrb_split_rows role 1)."""
    w32 = _final_attention_weights(model, torch.float32, device)
    return {k: (ops.split_rows(v, 1) if k.endswith("weight") else v) for k, v in w32.items()}


def _final_attention_weights(model, dtype: torch.dtype, device) -> dict:
    sd = model.state_dict()
    need = [f"linear{i}.weight" for i in range(1, 6)] + [f"linear{i}.bias" for i in range(1, 5)]
    for k in need:
        if k not in sd:
            raise _lib.NrbError(f"user encoder lacks {k}: not a FinalAttention state_dict")
    w = {}
    for k in need:
        t = sd[k].detach().to(device)
        w[k] = t.to(dtype).contiguous() if k.endswith("weight") else t.float().contiguous()
    return w


def _mark(stream) -> "torch.cuda.Event":
    ev = torch.cuda.Event(enable_timing=True)
    ev.record(stream)
    return ev


def _balanced_cuts(ho: np.ndarray, co: np.ndarray, n_imp: int, n_chunks: int, taper: bool = False) -> list:
    """Impression boundaries that split cost(i) = 2 * ho[i] + co[i] (table rows read up to impression i) evenly:
    the first i with cost(i) >= k / n_chunks of the total, by bisection on the two offset arrays -- a dozen
    element reads per cut instead of arithmetic over 2.4 M offsets (12 ms of host time the GPU would sit out)."""
    total = 2 * int(ho[n_imp]) + int(co[n_imp])
    cuts = {0, n_imp}
    fracs = [k / n_chunks for k in range(1, n_chunks)]
    if taper and n_chunks >= 2:  # the results of the LAST piece cross PCIe after all kernels are done: keep it small
        last = 1 / n_chunks
        while last > 1 / 32:
            last /= 2
            fracs.append(1 - last)
    for f in fracs:
        target = total * f
        lo, hi = 0, n_imp
        while lo < hi:
            mid = (lo + hi) // 2
            if 2 * int(ho[mid]) + int(co[mid]) < target:
                lo = mid + 1
            else:
                hi = mid
        cuts.add(lo)
    return sorted(cuts)


class ScoringEngine:
    """table + user encoder -> (scores, dense ranks) for CSR impressions, all on one GPU."""

    def __init__(self, news_embeddings: torch.Tensor, model: torch.nn.Module,
                 query_news_embeddings: Optional[torch.Tensor] = None, precision=None,
                 device: Optional[torch.device] = None, cache_table: bool = True):
        from .latent_attention import LatentAttentionModel

        self.device = _lib.require_device(device)
        self.dtype = precision_dtype(precision)
        self.split = precision_is_split(precision)
        self.model = model
        self.n_rows, self.dim = news_embeddings.shape
        self._streams = None
        self._staging: dict = {}
        self._staging_busy = False
        with torch.cuda.device(self.device):
            from .attention import NewAttention
            streamed = (not cache_table and not news_embeddings.is_cuda and query_news_embeddings is None
                        and not isinstance(model, (LatentAttentionModel, NewAttention))
                        and news_embeddings.dtype == torch.float32 and not self.split)
            if streamed:
                self._upload_and_transform_streamed(news_embeddings)
                return
            self.cand = resident_table(news_embeddings, self.dtype, self.device)
            src = news_embeddings if query_news_embeddings is None else query_news_embeddings
            hist_src = self.cand if query_news_embeddings is None else resident_table(src, self.dtype, self.device)
            self.prepare_user_encoder(hist_src)

    # -- host table -> device tables, copy engine and tensor cores overlapped --------------------------
    def _side_streams(self):
        if self._streams is None:
            self._streams = (torch.cuda.Stream(self.device), torch.cuda.Stream(self.device))
        return self._streams

    def _upload_and_transform_streamed(self, table_host: torch.Tensor, chunk_rows: int = 16384) -> None:
        """The fp32 host table crosses PCIe in row chunks on a copy stream while the previous chunk is
        converted and pushed through the per-row FinalAttention transform on the compute stream."""
        dev, n, d = self.device, self.n_rows, self.dim
        s_in, _ = self._side_streams()
        cur = torch.cuda.current_stream()
        fp = _model_fingerprint(self.model)
        if getattr(self, "_fa_weights_key", None) != fp:
            self._fa_weights = _final_attention_weights(self.model, self.dtype, dev)
            self._fa_weights_key = fp
        self._padded = None
        self._split_cand = None
        self.cand = torch.empty(n, d, dtype=self.dtype, device=dev)
        self.hist_x = torch.empty(n, d, dtype=self.dtype, device=dev)
        self.hist_e = torch.empty(n, d, dtype=self.dtype, device=dev)
        self.pool_mode = _lib.POOL_FINAL_ATTENTION
        direct = self.dtype == torch.float32
        stage = None if direct else [torch.empty(chunk_rows, d, dtype=torch.float32, device=dev) for _ in range(2)]
        free_ev = [None, None]
        s_in.wait_stream(cur)
        for k, r0 in enumerate(range(0, n, chunk_rows)):
            r1 = min(n, r0 + chunk_rows)
            b = k & 1
            with torch.cuda.stream(s_in):
                if direct:
                    self.cand[r0:r1].copy_(table_host[r0:r1], non_blocking=True)
                else:
                    if free_ev[b] is not None:
                        s_in.wait_event(free_ev[b])
                    stage[b][: r1 - r0].copy_(table_host[r0:r1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(s_in)
            cur.wait_event(ev)
            if not direct:
                ops.convert_rows(stage[b][: r1 - r0], self.dtype, out=self.cand[r0:r1])  # fp32 -> bf16 on the device
                free_ev[b] = torch.cuda.Event()
                free_ev[b].record(cur)
            ops.final_attention_rows(self.cand[r0:r1], self._fa_weights, self.dtype, x_out=self.hist_x[r0:r1],
                                     e_out=self.hist_e[r0:r1])

    def _host_staging(self, n_h: int, n_c: int, n_imp: int, narrow: bool):
        """Device-side staging of `score_host` (indices in, scores / ranks out); reallocated only to grow."""
        want = {"hi": (max(n_h, 1), torch.int32), "ci": (max(n_c, 1), torch.int32), "sc": (max(n_c, 1), torch.float32),
                "rk": (max(n_c, 1), torch.int32), "rk16": (max(n_c, 1) + 8 if narrow else 0, torch.int16),
                "ho": (n_imp + 1, torch.int64), "co": (n_imp + 1, torch.int64)}
        st, fresh = self._staging, False
        for k, (n, dt) in want.items():
            if k not in st or st[k].numel() < n:
                st[k] = torch.empty(n, dtype=dt, device=self.device)
                fresh = True
        return st, fresh

    def score_host(self, hist_idx: torch.Tensor, hist_off: torch.Tensor, cand_idx: torch.Tensor,
                   cand_off: torch.Tensor, scores_out: Optional[torch.Tensor] = None,
                   ranks_out: Optional[torch.Tensor] = None, n_chunks: int = 8):
        """HOST (ideally pinned) CSR arrays in, HOST scores / ranks out, pipelined over impression chunks:
        index H2D (copy stream) | fused score+rank kernel (compute stream) | result D2H (copy-out stream).

        hist_idx / cand_idx int32, hist_off / cand_off int64 [I+1] CPU tensors.  `ranks_out` may be int32 or int16:
        int16 ranks are narrowed on the device and cross PCIe at 2 bytes per candidate (6 instead of 8 bytes of
        results per candidate; a rank above 32767 raises OverflowError).

        The device staging belongs to the engine: one `score_host` call per engine at a time (the reference issues all
        GPU work from one thread, SURVEY 8b).  The call returns after its results have landed in the host buffers."""
        dev = self.device
        n_imp = hist_off.numel() - 1
        assert cand_off.numel() - 1 == n_imp, "Number of rows should be consistent"
        n_h, n_c = int(hist_off[-1]), int(cand_off[-1])
        assert n_h == hist_idx.numel() and n_c == cand_idx.numel(), \
            "Number of impressions should match length of impression list"
        if scores_out is None:
            scores_out = torch.empty(n_c, dtype=torch.float32).pin_memory()
        if ranks_out is None:
            ranks_out = torch.empty(n_c, dtype=torch.int32).pin_memory()
        with torch.cuda.device(dev):
            s_in, s_out = self._side_streams()
            cur = torch.cuda.current_stream()
            narrow = ranks_out.dtype == torch.int16
            # device staging owned by the engine (grow-only): nothing else ever touches it and every call ends with a
            # full synchronisation, so the copy-in stream may start at once -- this step's indices cross PCIe while
            # whatever the caller queued before (the per-row transform) still runs on the compute stream
            st, fresh = self._host_staging(n_h, n_c, n_imp, narrow)
            hi_d, ci_d, sc_d, rk_d, rk16_d = st["hi"], st["ci"], st["sc"], st["rk"], st["rk16"]
            ho_d, co_d = st["ho"][:n_imp + 1], st["co"][:n_imp + 1]
            flag = ops.new_err_flag(dev)
            if self._staging_busy:  # an earlier call was aborted half-way
                torch.cuda.synchronize(dev)
            elif fresh:  # new blocks may be recycled memory of work still queued on the compute stream
                s_in.wait_stream(cur)
            self._staging_busy = True
            # impression chunks balanced by the rows they read
            n_chunks = max(1, min(n_chunks, n_imp))
            bounds = _balanced_cuts(hist_off.numpy(), cand_off.numpy(), n_imp, n_chunks, taper=True)
            evs = []
            with torch.cuda.stream(s_in):
                ho_d.copy_(hist_off, non_blocking=True)
                co_d.copy_(cand_off, non_blocking=True)
            for i0, i1 in zip(bounds[:-1], bounds[1:]):
                h0, h1, c0, c1 = int(hist_off[i0]), int(hist_off[i1]), int(cand_off[i0]), int(cand_off[i1])
                with torch.cuda.stream(s_in):
                    hi_d[h0:h1].copy_(hist_idx[h0:h1], non_blocking=True)
                    ci_d[c0:c1].copy_(cand_idx[c0:c1], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(s_in)
                evs.append((i0, i1, c0, c1, ev))
            k_x, k_e, k_c = self._kernel_tables()
            trace = getattr(self, "_trace", None)  # diagnosis only (tools/e2e_timeline.py): [(label, event)]
            for i0, i1, c0, c1, ev in evs:
                cur.wait_event(ev)
                if trace is not None:
                    trace.append(("h2d_ready+wait %d" % i0, _mark(cur)))
                ops.score_rank(self.pool_mode, k_x, k_e, k_c, hi_d, ho_d[i0:i1 + 1], ci_d,
                               co_d[i0:i1 + 1], n_c, want_ranks=True, err_flag=flag, out_scores=sc_d, out_ranks=rk_d)
                if narrow and c1 > c0:
                    a0 = c0 - (c0 % 8)  # 16-byte aligned window (the overlap rewrites identical values)
                    ops.narrow_ranks(rk_d[a0:c1], rk16_d[a0:c1], flag)
                done = torch.cuda.Event(enable_timing=trace is not None)
                done.record(cur)
                s_out.wait_event(done)
                with torch.cuda.stream(s_out):
                    scores_out[c0:c1].copy_(sc_d[c0:c1], non_blocking=True)
                    ranks_out[c0:c1].copy_((rk16_d if narrow else rk_d)[c0:c1], non_blocking=True)
                    if trace is not None:
                        trace.append(("kernel_done %d" % i0, done))
                        trace.append(("d2h_done %d" % i0, _mark(s_out)))
            s_in.synchronize()
            s_out.synchronize()
            cur.synchronize()
            self._staging_busy = False
            ops.raise_on_index_error(flag, "score_host")
        return scores_out, ranks_out

    # -- tables as the fused kernel wants them -----------------------------------------------------------
    def _kernel_tables(self):
        """(hist_x, hist_e, cand) for `nrb_score_rank`, whose lanes own whole 16-byte vectors of a 512-byte multiple
        row.  The reference's usual widths (1024, 768, 512, 256) are that already and pass through untouched; any other
        width (384: bge-small, config.py:63) gets zero-padded copies of the three tables -- zero columns change no
        pooled value, dot product or norm, so scores and ranks are those of the logical width."""
        es = self.cand.element_size()
        d = self.cand.shape[1]
        if (d * es) % 512 == 0:
            return self.hist_x, self.hist_e, self.cand
        key = tuple((t.data_ptr(), t._version) for t in (self.hist_x, self.hist_e, self.cand) if t is not None)
        hit = getattr(self, "_padded", None)
        if hit is None or hit[0] != key:
            pad = lambda t: None if t is None else ops.pad_rows_for_kernel(t)
            hit = (key, (pad(self.hist_x), pad(self.hist_e), pad(self.cand)))
            self._padded = hit
        return hit[1]

    # -- per-row user-encoder transform (dense, once per table) --------------------------------
    def prepare_user_encoder(self, hist_src: torch.Tensor) -> None:
        from .attention import NewAttention
        from .latent_attention import LatentAttentionModel

        self._padded = None  # new tables may land at the old addresses: padded kernel copies are rebuilt
        self._split_cand = None  # likewise the split-bf16 copy of an fp32 table that `recommend` scores against

        if isinstance(self.model, NewAttention):
            # LayerNorm chain + exp(linear1): per-row, same exp-weighted pooling as FinalAttention
            self.hist_x, self.hist_e = self.model.row_tables(hist_src, self.dtype)
            self.pool_mode = _lib.POOL_FINAL_ATTENTION
        elif isinstance(self.model, LatentAttentionModel):
            # tokens are independent (SURVEY 3.2): run the block once per table row, then mean-pool
            fw = self.model.folded(self.dtype, self.device)
            rows = ops.latent_forward(fw, hist_src.view(self.n_rows, 1, self.dim), None,
                                      max_tokens=LATENT_MAX_TOKENS)
            self.hist_x = rows.view(self.n_rows, self.dim).to(self.dtype).contiguous()
            self.hist_e = None
            self.pool_mode = _lib.POOL_MEAN_L2
        else:
            # kernel-ready weights stay resident until a parameter changes (trainers update them per epoch)
            fp = _model_fingerprint(self.model)
            if getattr(self, "_fa_weights_key", None) != fp:
                self._fa_weights = (_final_attention_weights_split(self.model, self.device) if self.split else
                                    _final_attention_weights(self.model, self.dtype, self.device))
                self._fa_weights_key = fp
            if self.split:
                self.hist_x, self.hist_e = ops.final_attention_rows_split(hist_src, self._fa_weights)
            else:
                self.hist_x, self.hist_e = ops.final_attention_rows(hist_src, self._fa_weights, self.dtype)
            self.pool_mode = _lib.POOL_FINAL_ATTENTION

    # -- fused gather + pool + cosine + rank ---------------------------------------------------------
    def upload_impressions(self, hist_idx, hist_len, cand_idx, cand_len):
        n_imp = len(hist_len)
        assert n_imp == len(cand_len), "Number of rows should be consistent"  # data_model_helper.py:183
        h_off, n_h = _offsets(hist_len, self.device)
        c_off, n_c = _offsets(cand_len, self.device)
        assert n_c == len(cand_idx), "Number of impressions should match length of impression list"  # :186
        assert n_h == len(hist_idx), "history index length should match history_len_list"
        return (_as_i32(hist_idx, self.device), h_off, _as_i32(cand_idx, self.device), c_off, n_c)

    def score_device(self, hist_idx_d, hist_off_d, cand_idx_d, cand_off_d, n_cand: int, want_user=False,
                     want_ranks=True, err_flag=None, out_scores=None, out_ranks=None, cand_base=None,
                     blend_alpha: float = 1.0):
        with torch.cuda.device(self.device):
            k_x, k_e, k_c = self._kernel_tables()
            user, scores, ranks = ops.score_rank(self.pool_mode, k_x, k_e, k_c, hist_idx_d, hist_off_d,
                                                 cand_idx_d, cand_off_d, n_cand, want_user=want_user,
                                                 want_ranks=want_ranks, err_flag=err_flag, out_scores=out_scores,
                                                 out_ranks=out_ranks, cand_base=cand_base, blend_alpha=blend_alpha)
            if user is not None and user.shape[1] != self.cand.shape[1]:
                user = user[:, :self.cand.shape[1]].contiguous()  # drop the kernel's zero padding
            return user, scores, ranks

    def score(self, hist_idx, hist_len, cand_idx, cand_len, want_user=False, want_ranks=True, cand_base=None,
              blend_alpha: float = 1.0):
        """Host arrays in, device tensors out: (user|None, scores fp32, ranks int32|None).
        `cand_base` (fp32 per table row) + `blend_alpha` fuse the WeightedSumModel blend behind the cosine."""
        with torch.cuda.device(self.device):
            hi, ho, ci, co, n_c = self.upload_impressions(hist_idx, hist_len, cand_idx, cand_len)
            if cand_base is not None:
                cand_base = torch.as_tensor(cand_base, dtype=torch.float32).to(self.device).contiguous()
            return self.score_device(hi, ho, ci, co, n_c, want_user=want_user, want_ranks=want_ranks,
                                     cand_base=cand_base, blend_alpha=blend_alpha)

    def topk(self, scores_d: torch.Tensor, cand_off_d: torch.Tensor, k: int) -> torch.Tensor:
        """Positions of the k best candidates of every impression (int32 [I, k], -1 padded), from device scores."""
        with torch.cuda.device(self.device):
            return ops.topk_order(scores_d, cand_off_d, k)

    # -- whole-table retrieval ---------------------------------------------------------------------------------
    def _table_operand(self) -> torch.Tensor:
        """The bf16 GEMM operand `recommend` scores against: the table itself for bf16 engines, its [hi|lo|hi]
        split copy (cached until the tables are rebuilt) for fp32 / fp32x3 engines."""
        if self.cand.dtype == torch.bfloat16:
            return self.cand
        key = (self.cand.data_ptr(), self.cand._version)
        hit = getattr(self, "_split_cand", None)
        if hit is None or hit[0] != key:
            hit = (key, ops.split_rows(self.cand, 1))
            self._split_cand = hit
        return hit[1]

    def recommend_device(self, hist_idx_d: torch.Tensor, hist_off_d: torch.Tensor, k: int,
                         exclude_history: bool = True, err_flag: Optional[torch.Tensor] = None,
                         pool: Optional[torch.Tensor] = None, cand_base: Optional[torch.Tensor] = None,
                         blend_alpha: float = 1.0):
        """Device CSR history (int32 ids, int64 offsets [U + 1]) in, the k best table rows per user out:
        (rows int32 [U, k], scores fp32 [U, k]) on the device, see `ops.recommend` for the order and padding.

        The user vector is the one `score` pools; its score against row r is the cosine `score` would give r as a
        candidate.  With `exclude_history` a user's own history rows are never returned.  `pool` (device int32 row
        ids, strictly ascending) restricts the rows; `cand_base` (device fp32 per table row) + `blend_alpha` blend the
        baseline in as `score` does, users with an empty history getting the baseline alone.  fp32 and fp32x3 engines
        score on split-bf16 tensor-core operands (the FFMA GEMM has no top-k epilogue)."""
        ops._recommend_args(self.dim, k)
        ops._recommend_pool_args(self.n_rows, hist_off_d.numel() - 1, pool, cand_base, None)
        with torch.cuda.device(self.device):
            flag = err_flag if err_flag is not None else ops.new_err_flag(self.device)
            n_imp = hist_off_d.numel() - 1
            zeros = torch.zeros(n_imp + 1, dtype=torch.int64, device=self.device)
            empty = torch.zeros(1, dtype=torch.int32, device=self.device)
            k_x, k_e, k_c = self._kernel_tables()
            user, _, _ = ops.score_rank(self.pool_mode, k_x, k_e, k_c, hist_idx_d, hist_off_d, empty, zeros, 0,
                                        want_user=True, want_ranks=False, err_flag=flag)
            if user.shape[1] != self.dim:
                user = user[:, :self.dim].contiguous()  # drop the kernel's zero padding: logical rows and width
            excl = (hist_idx_d, hist_off_d) if exclude_history else (None, None)
            rows, scores = ops.recommend(self.cand, user, k, table_op=self._table_operand(), excl_idx=excl[0],
                                         excl_off=excl[1], err_flag=flag, pool=pool, cand_base=cand_base,
                                         blend_alpha=blend_alpha, hist_off=hist_off_d)
            if err_flag is None:
                ops.raise_on_index_error(flag, "recommend")
            return rows, scores

    def recommend(self, hist_idx, hist_len, k: int, exclude_history: bool = True, pool=None, cand_base=None,
                  blend_alpha: float = 1.0):
        """Host history arrays (`history_rev_ind_array[0]`, `history_len_list`) in: the k best rows of the table for
        each user, (rows int32 [U, k], scores fp32 [U, k]) on the device.  `pool`: host row ids (any order,
        duplicates allowed) or a bool mask over the table, see `host_pool`; `cand_base`: fp32 per table row."""
        ops._recommend_args(self.dim, k)
        pool_np = None if pool is None else host_pool(pool, self.n_rows)
        base_np = None if cand_base is None else host_base(cand_base, self.n_rows)
        with torch.cuda.device(self.device):
            h_off, n_h = _offsets(hist_len, self.device)
            assert n_h == len(hist_idx), "history index length should match history_len_list"
            pool_d = None if pool_np is None else torch.from_numpy(pool_np).to(self.device)
            base_d = None if base_np is None else torch.from_numpy(base_np).to(self.device)
            return self.recommend_device(_as_i32(hist_idx, self.device), h_off, k, exclude_history=exclude_history,
                                         pool=pool_d, cand_base=base_d, blend_alpha=blend_alpha)

    def user_vectors(self, hist_idx, hist_len) -> torch.Tensor:
        """get_final_attention_eval: fp32 [I, d] user vectors (device)."""
        with torch.cuda.device(self.device):
            n_imp = len(hist_len)
            h_off, n_h = _offsets(hist_len, self.device)
            assert n_h == len(hist_idx)
            zeros = torch.zeros(n_imp + 1, dtype=torch.int64, device=self.device)
            empty = torch.zeros(1, dtype=torch.int32, device=self.device)
            k_x, k_e, k_c = self._kernel_tables()
            user, _, _ = ops.score_rank(self.pool_mode, k_x, k_e, k_c,
                                        _as_i32(hist_idx, self.device), h_off, empty, zeros, 0, want_user=True,
                                        want_ranks=False)
            return user if user.shape[1] == self.cand.shape[1] else user[:, :self.cand.shape[1]].contiguous()


def host_pool(pool, n_rows: int) -> np.ndarray:
    """A host pool as `ops.recommend` takes it: a bool mask over the n_rows table rows -> the rows it selects, or row
    ids in any order with duplicates -> the distinct ids ascending (int32).  Ids outside [0, n_rows) raise IndexError."""
    p = np.asarray(pool)
    if p.dtype == np.bool_:
        if p.shape != (n_rows,):
            raise ValueError(f"a boolean pool must be a mask over the {n_rows} table rows, got shape {p.shape}")
        return np.flatnonzero(p).astype(np.int32)
    if p.ndim != 1 or (p.size and not np.issubdtype(p.dtype, np.integer)):
        raise ValueError("a pool must be a 1-D array of integer row ids or a boolean mask")
    ids = np.unique(p.astype(np.int64))
    if ids.size and (ids[0] < 0 or ids[-1] >= n_rows):
        raise IndexError(f"pool: row id out of range for a table of {n_rows} rows")
    return ids.astype(np.int32)


def host_base(cand_base, n_rows: int) -> np.ndarray:
    """A host per-row baseline (one fp32 score per table row, e.g. `get_classification_preds`)."""
    b = np.ascontiguousarray(np.asarray(cand_base, dtype=np.float32))
    if b.shape != (n_rows,):
        raise ValueError(f"the baseline must have one score per table row ({n_rows}), got shape {b.shape}")
    return b


_engine_cache: dict = {}


def _model_fingerprint(model: torch.nn.Module) -> tuple:
    return tuple((k, v.data_ptr(), v._version) for k, v in model.state_dict(keep_vars=True).items())


def cached_engine(news_embeddings: torch.Tensor, model: torch.nn.Module,
                  query_news_embeddings: Optional[torch.Tensor] = None, precision=None) -> ScoringEngine:
    """Engines are expensive (table upload + dense row transform): reuse them while the table and
    the weights are unchanged (the trainers call the hot path every epoch with new weights)."""
    q = query_news_embeddings
    key = (id(news_embeddings), news_embeddings.data_ptr(), news_embeddings._version,
           None if q is None else (id(q), q.data_ptr(), q._version), id(model), _model_fingerprint(model),
           str(precision_dtype(precision)), precision_is_split(precision))
    hit = _engine_cache.get(key)
    if hit is not None:
        # id / data_ptr / _version can all repeat after the table is freed (or be untouched by a numpy-side
        # edit of a from_numpy table's storage owner): the entry is valid only for the very same live objects
        eng, t_ref, q_ref = hit
        if t_ref() is news_embeddings and (q is None or (q_ref is not None and q_ref() is q)):
            return eng
    _engine_cache.clear()
    eng = ScoringEngine(news_embeddings, model, q, precision=precision)
    try:
        _engine_cache[key] = (eng, weakref.ref(news_embeddings), None if q is None else weakref.ref(q))
    except TypeError:
        pass
    return eng
