"""Whole-table retrieval at MIND-large scale: fused tensor-core GEMM + top-k (nrb_recommend) vs the unfused path, and
retrieval from a pool with the classification-baseline blend (nrb_recommend_pool_blend).

    python tools/recommend_bench.py [--users 65536] [--ks 10,32] [--iters 5] [--pool-k 10] [--out FILE]

Workload: the MIND-large table (161,013 x 1024, bf16, synthetic FinalAttention weights as in bench.py), U users with
bench.py's history distribution (H ~ clip(Geom(1/32), 1, 50)), history excluded.  Per k it reports, from CUDA events
after warm-up:
  * ms per call: pooling (score_rank user vectors), fused recommend (user operand + row norms + history sort + GEMM
    with top-k epilogue + merge), and a kernel-level split of the fused call from a separate torch.profiler pass;
  * executed TFLOP/s of the fused GEMM (2 U N d / t) and its fraction of the sustained bf16 peak of
    MEASURED_PEAKS.json (bench.py's fallback figure when the file is absent);
  * the unfused path in the same process: nrb_linear to fp32 scores in user chunks, scale by the row norms, mask
    history, torch.topk; its time and the number of users whose row lists differ from the fused result.
Then, at k = --pool-k, four legs of the fused call timed back to back in the same process ("pool_blend"): plain,
pool = a random N/8 of the rows, blend (baseline for every row, alpha 0.7, the bench's users all have a history), and
pool + blend; each with ms per call and the executed TFLOP/s of the call, 2 U n_pool d / t (n_pool = N without a
pool).  The legs run after each other in rounds (plain, pool, blend, pool + blend, repeated --rounds times) and report
the median, so that a drift of the clocks over the run reaches every leg alike.
The GPU name and power limit come from a read-only nvidia-smi query in the same run.  Needs a B200.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (measured_peaks, make_device_impressions, the bench's table shape)
from news_recommendation_project_v2_b200 import _lib, ops, synthetic as syn  # noqa: E402
from news_recommendation_project_v2_b200.engine import ScoringEngine  # noqa: E402
from news_recommendation_project_v2_b200.modeling_utils import FinalAttention  # noqa: E402


def gpu_info() -> dict:
    q = "name,power.limit,power.max_limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        vals = [v.strip() for v in out.split(",")]
        return dict(zip(q.split(","), vals))
    except Exception as e:  # noqa: BLE001
        return {"error": str(e), "name": torch.cuda.get_device_name(0)}


def timed(fn, iters: int) -> float:
    """ms per call from CUDA events around `iters` back-to-back calls (after the caller's warm-up)."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def unfused(user, table_pad, inv_norm_pad, n_rows, hist_idx, h_off, k, chunk):
    """nrb_linear -> fp32 scores per user chunk, cosine scaling, history masked to -inf, torch.topk."""
    U = user.shape[0]
    un = (user / user.norm(dim=1, keepdim=True).clamp_min(1e-8)).to(torch.bfloat16)
    rows = torch.empty(U, k, dtype=torch.int64, device=user.device)
    vals = torch.empty(U, k, dtype=torch.float32, device=user.device)
    lens = (h_off[1:] - h_off[:-1])
    for i0 in range(0, U, chunk):
        i1 = min(U, i0 + chunk)
        s = ops.linear(un[i0:i1].contiguous(), table_pad, out_dtype=torch.float32)
        s.mul_(inv_norm_pad)
        s[:, n_rows:] = -float("inf")
        h0, h1 = int(h_off[i0]), int(h_off[i1])
        owner = torch.repeat_interleave(torch.arange(i1 - i0, device=user.device), lens[i0:i1])
        s[owner, hist_idx[h0:h1].long()] = -float("inf")
        v, r = torch.topk(s, k, dim=1)
        rows[i0:i1], vals[i0:i1] = r, v
    return rows, vals


def kernel_split(fn) -> dict:
    """ms of each kernel of one fused call (torch.profiler, its own pass)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out: dict = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.name
        key = ("gemm_topk" if "gemm_tc_kernel" in name else "merge" if "merge_kernel" in name else
               "user_operand" if "user_operand" in name else "row_norms" if "row_scale" in name else
               "history_sort" if "sort_excl" in name else "pool_gather" if "pool_gather" in name else None)
        if key is None:
            continue
        out[key] = out.get(key, 0.0) + ev.device_time / 1000.0
    return {k: round(v, 4) for k, v in out.items()}


def pool_blend_legs(eng, user, hist_idx, h_off, k, iters, warmup, rounds, flag) -> dict:
    """ms per call and executed TFLOP/s of plain / pool N/8 / blend / pool + blend, alternated over `rounds`."""
    n_rows, d = eng.cand.shape
    U = user.shape[0]
    g = torch.Generator(device=user.device).manual_seed(99)
    pool = torch.sort(torch.randperm(n_rows, generator=g, device=user.device)[:n_rows // 8])[0].to(torch.int32)
    base = torch.rand(n_rows, generator=g, device=user.device)  # a classification probability per row
    legs = {"plain": {}, "pool_n_over_8": dict(pool=pool), "blend": dict(cand_base=base, blend_alpha=0.7),
            "pool_n_over_8_blend": dict(pool=pool, cand_base=base, blend_alpha=0.7)}
    fns = {name: (lambda kw=kw: ops.recommend(eng.cand, user, k, excl_idx=hist_idx, excl_off=h_off, err_flag=flag,
                                               hist_off=h_off, **kw)) for name, kw in legs.items()}
    for fn in fns.values():
        for _ in range(warmup):
            fn()
    times = {name: [] for name in fns}
    for _ in range(rounds):
        for name, fn in fns.items():
            times[name].append(timed(fn, iters))
    out = {"k": k, "n_pool": int(pool.numel()), "rounds": rounds, "iters_per_round": iters, "legs": {}}
    for name, ts in times.items():
        t = sorted(ts)[len(ts) // 2]
        cols = int(pool.numel()) if "pool" in legs[name] else n_rows
        out["legs"][name] = {"ms": round(t, 4), "ms_all_rounds": [round(x, 4) for x in ts],
                             "tflops": round(2.0 * U * cols * d / (t * 1e-3) / 1e12, 1),
                             "kernels_ms": kernel_split(fns[name])}
        print(f"pool/blend k={k} {name}: {t:.3f} ms, {out['legs'][name]['tflops']} TFLOP/s", file=sys.stderr)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=65536)
    ap.add_argument("--ks", default="10,32")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--chunk", type=int, default=4096, help="users per unfused GEMM chunk")
    ap.add_argument("--pool-k", type=int, default=10, help="k of the pool / blend legs")
    ap.add_argument("--rounds", type=int, default=5, help="rounds over the pool / blend legs")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    dev = _lib.require_device()
    info = gpu_info()
    n_rows, d, hidden, h_max = bench.N_ROWS, bench.DIM, bench.HIDDEN, bench.H_MAX
    U = a.users
    model = FinalAttention(d, hidden, precision="bf16")
    model.load_state_dict(syn.make_final_attention_state_dict(d, hidden, seed=1234))
    table = syn.make_table(n_rows, d, seed=1234)
    eng = ScoringEngine(table, model.eval(), precision="bf16")
    hist_idx, h_off, *_ = bench.make_device_impressions(U, n_rows, h_max, 4321, dev)
    n_hist = int(h_off[-1])

    zeros = torch.zeros(U + 1, dtype=torch.int64, device=dev)
    empty = torch.zeros(1, dtype=torch.int32, device=dev)
    k_x, k_e, k_c = eng._kernel_tables()

    def pool():
        return ops.score_rank(eng.pool_mode, k_x, k_e, k_c, hist_idx, h_off, empty, zeros, 0, want_user=True,
                              want_ranks=False)[0]

    user = pool()
    for _ in range(a.warmup):
        pool()
    t_pool = timed(pool, a.iters)

    # unfused operands: table padded to a multiple of 32 rows (nrb_linear's N), row norms in fp32
    n_pad = (n_rows + 31) // 32 * 32
    table_pad = torch.zeros(n_pad, d, dtype=torch.bfloat16, device=dev)
    table_pad[:n_rows] = eng.cand
    inv = torch.full((n_pad,), float("nan"), device=dev)
    inv[:n_rows] = 1.0 / eng.cand.float().norm(dim=1).clamp_min(1e-8)

    peaks = bench.measured_peaks()
    results = {"workload": {"table_rows": n_rows, "dim": d, "users": U, "history_max": h_max, "sum_history": n_hist,
                            "table_dtype": "bf16", "encoder": "FinalAttention (synthetic weights)",
                            "exclude_history": True},
               "gpu": info, "peaks": peaks, "iters": a.iters, "warmup": a.warmup, "pool_ms": round(t_pool, 4),
               "by_k": {}}
    flops = 2.0 * U * n_rows * d
    flag = ops.new_err_flag(dev)  # checked once at the end: no host synchronisation inside the timed calls
    for k in [int(x) for x in a.ks.split(",")]:
        def fused():
            return ops.recommend(eng.cand, user, k, excl_idx=hist_idx, excl_off=h_off, err_flag=flag)
        for _ in range(a.warmup):
            fused()
        t_fused = timed(fused, a.iters)
        split = kernel_split(fused)
        r_f, s_f = fused()

        def unf():
            return unfused(user, table_pad, inv, n_rows, hist_idx, h_off, k, a.chunk)
        unf()
        t_unf = timed(unf, max(1, a.iters // 2))
        r_u, s_u = unf()
        diff_rows = int((r_f.long() != r_u).any(dim=1).sum())
        # lists that differ only by the order of equal scores / rows whose scores differ by float rounding
        diff_sets = int((torch.sort(r_f.long(), dim=1)[0] != torch.sort(r_u, dim=1)[0]).any(dim=1).sum())
        max_score_diff = float((s_f - s_u).abs().max())
        t_gemm = split.get("gemm_topk")
        results["by_k"][str(k)] = {
            "fused_ms": round(t_fused, 4), "pool_plus_fused_ms": round(t_pool + t_fused, 4),
            "kernels_ms": split,
            "gemm_topk_tflops": round(flops / (t_gemm * 1e-3) / 1e12, 1) if t_gemm else None,
            "gemm_topk_frac_sustained_bf16": round(flops / (t_gemm * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"], 3)
            if t_gemm else None,
            "fused_call_tflops": round(flops / (t_fused * 1e-3) / 1e12, 1),
            "unfused_ms": round(t_unf, 4), "unfused_chunk_users": a.chunk,
            "speedup_fused_vs_unfused": round(t_unf / t_fused, 2),
            "users_with_different_lists": diff_rows, "users_with_different_row_sets": diff_sets,
            "max_abs_score_diff_fused_vs_unfused": max_score_diff,
        }
        print(f"k={k}: fused {t_fused:.3f} ms {split}, unfused {t_unf:.3f} ms, lists differ for {diff_rows} users",
              file=sys.stderr)
    results["pool_blend"] = pool_blend_legs(eng, user, hist_idx, h_off, a.pool_k, a.iters, a.warmup, a.rounds, flag)
    ops.raise_on_index_error(flag, "recommend_bench")
    line = json.dumps(results)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(results, indent=1) + "\n")


if __name__ == "__main__":
    main()
