#!/usr/bin/env python
"""Headline benchmark: impressions/sec scored (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of scripts/eval.py's FinalAttentionComponent.transform over the rank's shard
of a MIND-large-shaped synthetic evaluation set (BASELINE.json configs[3]; SURVEY.md 8d):
  per step = FinalAttention per-row transform of the WHOLE table (5 tcgen05 GEMMs, hoisted from the
             reference's per-history-slot MLPs -- it is redone every step so that no reference
             work is skipped) + ONE fused gather/pool/cosine/dense-rank launch over all impressions.

Keys of the JSON line (one line, rank 0):
`value`   : impressions/s with the table, weights and CSR indices already resident in HBM.  WEAK scaling:
            every rank scores its own --impressions (2.4 M) against its replica of the table, no data-path
            collective (impressions are independent units).
`e2e`     : the same step through the public host API (ScoringEngine) with HOST buffers: every step copies its CSR
            indices H2D from pinned memory and its scores + ranks D2H; the engine (table + transformed tables) stays
            resident across steps exactly as `cached_engine` keeps it for repeated calls on the same table object.
            `e2e.cold` also re-uploads the pinned fp32 table every step (a first call on a new table).
            `e2e.link_probe`: H2D / D2H GB/s per rank with every rank copying at once (names the multi-GPU limiter).
`roofline`: the fused score/rank kernel against the measured HBM copy bandwidth.
`strong`  : (N > 1) BASELINE configs[3] as written: 2.4 M impressions TOTAL partitioned over the ranks
            (cost-balanced contiguous blocks), the per-row transform partitioned too (each rank transforms
            N/world rows and the transformed rows are all-gathered over NVLink), raw table replicated.
`cfg5`    : (N > 1) BASELINE configs[4]: history <= 200, d=1024, 1024 latents, 1.25 M table rows per GPU
            (10 M at 8 GPUs) row-sharded: per-shard latent transform + all-gather + local scoring.
`stage_a` : latent-attention pooling (BASELINE configs[2] shape) on a 32,768-item chunk, `cfg3`: the full
            1,000,000-item job streamed in 65,536-item chunks; news/s and fraction of the measured bf16 peak.
`cfg2`    : BASELINE configs[1]: 1,024 impressions (launch-latency bound), eager and CUDA-graph replay.
`fp32`    : the rank-exact fp32 path (FFMA row transform + fp32 tables) on the headline workload.
`cpu_baseline` / `reference_gpu`: the UNMODIFIED reference (oracle/_ref, see oracle/build_ref.py) on the host
            cores, and the same reference code with DEVICE=cuda on this B200 (the same-box torch number).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from news_recommendation_project_v2_b200 import synthetic as syn  # noqa: E402

METRIC = "impressions_per_sec_scored"
UNIT = "impressions/s"

# MIND-large-shaped workload (SURVEY.md 8d cfg 4)
N_ROWS, DIM, HIDDEN, H_MAX = 161_013, 1024, 4096, 50
E2E_CHUNKS = int(os.environ.get("NRB200_E2E_CHUNKS", "8"))  # impression chunks of the host-buffer pipeline
WORKLOAD = ("MIND-large-shaped eval (BASELINE configs[3]): FinalAttention user encoder, "
            "gather+pool+cosine+dense-rank")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline (and of --workload cfg5); the secondary legs reported under "
                         "their own keys keep their own step counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["native", "reference", "reference-gpu"], default="native")
    ap.add_argument("--impressions", type=int, default=2_400_000, help="impressions per rank per step")
    ap.add_argument("--precision", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--no-stage-a", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--no-extras", action="store_true",
                    help="profiling runs only: skip cfg2 / cfg3 / fp32 / reference_gpu / strong / cfg5 legs")
    ap.add_argument("--only-stage-a", action="store_true", help="profiling runs only: latent-attention pooling leg")
    ap.add_argument("--ref-sample", type=int, default=1024,
                    help="impressions per step of the CPU reference arm (cpu_baseline of the native arm: 4x, once)")
    ap.add_argument("--workload", choices=["cfg4", "cfg5"], default="cfg4",
                    help="cfg4 = headline (replicated table); cfg5 = long-history stress, row-sharded table")
    ap.add_argument("--table-rows", type=int, default=0, help="cfg5: total table rows (default 1.25 M per GPU)")
    ap.add_argument("--gather", choices=["auto", "p2p", "dma", "nccl", "nvls", "none"], default="auto",
                    help="cfg5 / strong: all-gather implementation (auto = nvls when NVLink multicast is available, "
                         "else dma; none = transform only, for diagnosis: results invalid)")
    ap.add_argument("--chunk-rows", type=int, default=0, help="cfg5: table rows transformed + pushed per chunk")
    ap.add_argument("--strong-chunks", type=int, default=4, help="strong leg: chunks per rank of the row transform")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's scores and dense ranks of the last timed step (a fixed, "
                         "seeded sample of whole impressions, at most 64 MB) as DIR/<name>.npy, so that two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native path (--impl native)")
    if args.dump_outputs and args.only_stage_a:
        ap.error("--dump-outputs writes the headline step's outputs, which --only-stage-a does not run")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    # fallback stated in /opt/skills/guides/B200_PROFILING.md
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
def make_device_impressions(n_imp: int, n_rows: int, h_max: int, seed: int, device, cand: str = "large"):
    """cfg-4 shaped CSR impressions generated on the device (SURVEY 8d): H ~ clip(Geom(1/32),1,h_max),
    C ~ clip(round(LogNormal(ln 30, 0.7)), 2, 300) ('large') or UniformInt[3,7] ('small'), uniform row ids."""
    g = torch.Generator(device=device).manual_seed(seed)
    hist_len = torch.empty(n_imp, device=device).geometric_(1.0 / 32.0, generator=g).clamp_(1, h_max).to(torch.int64)
    if cand == "large":
        cand_len = torch.empty(n_imp, device=device).log_normal_(float(np.log(30.0)), 0.7, generator=g).round_() \
            .clamp_(2, 300).to(torch.int64)
    else:
        cand_len = torch.randint(3, 8, (n_imp,), generator=g, device=device, dtype=torch.int64)
    h_off = torch.zeros(n_imp + 1, dtype=torch.int64, device=device)
    c_off = torch.zeros(n_imp + 1, dtype=torch.int64, device=device)
    torch.cumsum(hist_len, 0, out=h_off[1:])
    torch.cumsum(cand_len, 0, out=c_off[1:])
    n_h, n_c = int(h_off[-1]), int(c_off[-1])
    hist_idx = torch.randint(0, n_rows, (n_h,), generator=g, device=device, dtype=torch.int32)
    cand_idx = torch.randint(0, n_rows, (n_c,), generator=g, device=device, dtype=torch.int32)
    return hist_idx, h_off, cand_idx, c_off, hist_len.to(torch.int32), cand_len.to(torch.int32), n_h, n_c


def make_device_labels(c_off: torch.Tensor, seed: int, device) -> torch.Tensor:
    """int8 click labels per candidate (SURVEY 8d): one uniformly placed positive per impression, the others
    Bernoulli(0.04), at least one negative (evaluation.py:49 needs both classes)."""
    g = torch.Generator(device=device).manual_seed(seed)
    n_imp = c_off.numel() - 1
    cnt = c_off[1:] - c_off[:-1]
    n_c = int(c_off[-1])
    lab = (torch.rand(n_c, generator=g, device=device) < 0.04).to(torch.int8)
    pos = c_off[:-1] + (torch.rand(n_imp, generator=g, device=device, dtype=torch.float64) * cnt.double()).long() \
        .minimum(cnt - 1)
    lab[pos] = 1
    seg = torch.repeat_interleave(torch.arange(n_imp, device=device), cnt)
    tot = torch.zeros(n_imp, dtype=torch.int64, device=device).index_add_(0, seg, lab.long())
    full = torch.nonzero(tot == cnt).flatten()  # all positive: clear the slot after the forced positive
    if full.numel():
        nxt = c_off[:-1][full] + (pos[full] - c_off[:-1][full] + 1) % cnt[full]
        lab[nxt] = 0
    return lab


DUMP_MAX_CANDIDATES = 4_000_000  # scores + ranks in float32: 32 MB


def dump_outputs(out_dir: str, scores: torch.Tensor, ranks: torch.Tensor, c_off: torch.Tensor):
    """Write what a step returned to its caller -- per-candidate scores and dense ranks -- for whole impressions
    drawn in a seeded random order until DUMP_MAX_CANDIDATES candidates are taken, stored in ascending impression
    order.  The inputs are seeded, so two builds run with the same arguments dump the same positions."""
    n_imp = c_off.numel() - 1
    counts = (c_off[1:] - c_off[:-1]).cpu()
    order = torch.randperm(n_imp, generator=torch.Generator().manual_seed(0))
    keep = int(torch.searchsorted(torch.cumsum(counts[order], 0), DUMP_MAX_CANDIDATES, right=True))
    imp = order[:max(keep, 1)].sort().values
    cnt = counts[imp]
    first = c_off[:-1].cpu()[imp]
    local = torch.arange(int(cnt.sum())) - torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    pos = (torch.repeat_interleave(first, cnt) + local).to(scores.device)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"scores": scores[pos].float(), "ranks": ranks[pos].float(),
              "impressions": imp.double(), "candidates_per_impression": cnt.double()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())
    print("bench: wrote %s/{%s}.npy (%d impressions, %d candidates)" % (out_dir, ",".join(arrays), imp.numel(),
                                                                      pos.numel()), file=sys.stderr, flush=True)


def _ev():
    return torch.cuda.Event(enable_timing=True)


class Dist:
    """rank / world / device + barrier + MAX-reduction, with or without a process group."""

    def __init__(self, need_group: bool = False):
        import torch.distributed as dist

        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1 or need_group:
            if self.world == 1:
                os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
                os.environ.setdefault("MASTER_PORT", "29533")
                os.environ.setdefault("RANK", "0")
                os.environ.setdefault("WORLD_SIZE", "1")
            # NCCL's INFO lines (communicator size, transport, NVLS) go to stderr: stdout carries the JSON line only
            os.environ["NCCL_DEBUG"] = os.environ.get("NRB200_NCCL_DEBUG", "INFO")
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
            dist.init_process_group("nccl", device_id=self.dev)

    @property
    def grouped(self) -> bool:
        return self.dist.is_initialized()

    def barrier(self):
        torch.cuda.synchronize()
        if self.grouped and self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_ms(self, ms: float) -> float:
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.grouped and self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather_floats(self, v: float) -> list:
        t = torch.tensor([v], dtype=torch.float64, device=self.dev)
        if self.grouped and self.world > 1:
            out = [torch.zeros_like(t) for _ in range(self.world)]
            self.dist.all_gather(out, t)
            return [float(x.item()) for x in out]
        return [float(v)]

    def close(self):
        if self.grouped:
            self.dist.barrier()
            self.dist.destroy_process_group()


def _stdout_to_stderr_for_native_libs():
    """NCCL (NCCL_DEBUG=INFO) and other native code print on fd 1; the contract wants ONE JSON line there.
    Point fd 1 at stderr and hand Python a private duplicate of the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w")


def run_native(args):
    from news_recommendation_project_v2_b200 import _lib, hostmem, ops
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention

    _stdout_to_stderr_for_native_libs()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = hostmem.bind_to_gpu_numa(local)  # before any pinned allocation: first touch places the staging buffers
    D = Dist()
    rank, world, dev = D.rank, D.world, D.dev
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    _lib.require_device(dev)
    lib = _lib.load()
    peaks = measured_peaks()
    if args.only_stage_a:
        print(json.dumps({"stage_a": bench_stage_a(dev, peaks, args)}), flush=True)
        return
    dtype = torch.bfloat16 if args.precision == "bf16" else torch.float32
    es = 2 if dtype == torch.bfloat16 else 4

    # ---- synthetic inputs (random-init weights of the reference architecture) -------------------
    torch.manual_seed(1234)
    model = FinalAttention(DIM, HIDDEN, precision=args.precision).eval()
    model.load_state_dict(syn.make_final_attention_state_dict(DIM, HIDDEN, seed=1234))
    model.to(dev)  # the reference's factory does .to(DEVICE) (modeling_utils.py:274-279)
    table_host = syn.make_table(N_ROWS, DIM, seed=1234).pin_memory()  # fp32, L2-normalised (save_emb.py)
    n_imp = args.impressions
    hist_idx, h_off, cand_idx, c_off, hist_len, cand_len, n_h, n_c = make_device_impressions(
        n_imp, N_ROWS, H_MAX, 1234 + rank, dev)

    eng = ScoringEngine(table_host, model, precision=args.precision, device=dev)
    hist_src = eng.cand
    scores = torch.empty(n_c, dtype=torch.float32, device=dev)
    ranks = torch.empty(n_c, dtype=torch.int32, device=dev)
    flag = ops.new_err_flag(dev)

    def step(kernel_events=None):
        eng.prepare_user_encoder(hist_src)  # dense per-row transform (tcgen05)
        if kernel_events is not None:
            kernel_events[0].record()
        eng.score_device(hist_idx, h_off, cand_idx, c_off, n_c, want_ranks=True, err_flag=flag,
                         out_scores=scores, out_ranks=ranks)
        if kernel_events is not None:
            kernel_events[1].record()

    for _ in range(max(args.warmup, 3)):
        step()
    D.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = lib.nrb_kernel_launches()
    kev = [(_ev(), _ev()) for _ in range(args.steps)]
    t0, t1 = _ev(), _ev()
    D.barrier()
    t0.record()
    for i in range(args.steps):
        step(kev[i])
    t1.record()
    D.barrier()
    ms_total = t0.elapsed_time(t1)
    launches = lib.nrb_kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ops.raise_on_index_error(flag, "bench")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, scores, ranks, c_off)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    ms_step = D.max_ms(ms_total) / args.steps
    value = n_imp * world / (ms_step * 1e-3)

    # ---- roofline of the dominant kernel (fused score/rank): algorithmic bytes / launch ---------
    r = 2  # FinalAttention reads x and exp(logit) per history slot
    alg_bytes = (r * n_h + n_c) * DIM * es + 4 * (n_h + n_c) + 8 * n_c
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_note = None, "no ncu capture for this configuration"
    tpath = os.path.join(ROOT, "profiles", "score_rank_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            # the capture is only valid for the configuration it was taken on (keyed by the algorithmic bytes)
            if int(tj.get("algorithmic_bytes_per_launch", -1)) == int(alg_bytes):
                traffic, traffic_note = tj.get("dram_bytes_per_launch"), tj.get("source", "ncu --set full")
            else:
                traffic_note = "profiles/score_rank_traffic.json was captured on another configuration"
        except Exception:
            pass
    roofline = {"bound": "hbm", "kernel": "score_rank_kernel", "achieved": round(achieved, 1),
                "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(achieved / peaks["hbm_gbs"], 4),
                "traffic": traffic, "traffic_source": traffic_note, "peak_source": peaks["source"],
                "kernel_ms": round(kernel_ms, 3), "algorithmic_bytes_per_launch": int(alg_bytes),
                "share_of_step": round(kernel_ms / ms_step, 4),
                "note": "peak = measured COPY bandwidth (half reads, half writes); this kernel is 99.8 % reads and "
                        "~3 % of its algorithmic bytes are L2 hits, so frac can exceed 1"}

    out = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "impressions_per_gpu": n_imp, "table_rows": N_ROWS, "dim": DIM, "hidden": HIDDEN,
                   "history_max": H_MAX, "sum_history": n_h, "sum_candidates": n_c,
                   "sharding": "impressions sharded, table replicated, no data-path collective (weak: every rank "
                               "scores its own impressions; the `strong` key holds 2.4 M impressions TOTAL)",
                   "l2": "inputs_exceed_l2 (tables %.2f GB + indices %.2f GB per step)" %
                         (3 * N_ROWS * DIM * es / 1e9, 4 * (n_h + n_c) / 1e9)},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "clocks": clocks,
    }

    extras = not args.no_extras

    def guarded(key, fn, *a):
        """An extra leg must never cost the headline line: its failure is recorded under its own key."""
        try:
            out[key] = fn(*a)
        except Exception as exc:  # pragma: no cover - reported, not hidden
            import traceback

            traceback.print_exc(file=sys.stderr)
            out[key] = {"error": repr(exc)[:400]}
            try:
                torch.cuda.synchronize()
            except Exception:
                pass

    def run_e2e():
        if not args.no_e2e:
            out["e2e"] = leg_e2e(args, D, eng, model, table_host, hist_idx, h_off, cand_idx, c_off, n_imp, n_h, n_c,
                                 scores, ranks, numa)
        else:
            out["e2e"] = {"value": 0.0, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "steps": 0}

    if world > 1:
        run_e2e()
    if world > 1 and extras:
        guarded("strong", leg_strong, args, D, model, eng, ms_step, peaks)
        del eng
        torch.cuda.empty_cache()
        guarded("cfg5", leg_cfg5, args, D, peaks)
    if world == 1:
        # the tensor-core legs run straight after the headline, before the long host-buffer legs heat the package
        # further: under sw_power_cap the SM clock (and with it TFLOP/s) moves a few per cent with the temperature
        if not args.no_stage_a:
            guarded("stage_a", bench_stage_a, dev, peaks, args)
        if extras and not args.no_stage_a:
            guarded("cfg3", leg_cfg3, dev, peaks)
        run_e2e()
        if extras:
            if not args.no_stage_a and "cfg3" in out:
                if "error" not in out["cfg3"]:
                    try:
                        out["cfg3"]["e2e"] = leg_cfg3_e2e(dev)
                    except Exception as exc:  # pragma: no cover
                        out["cfg3"]["e2e"] = {"error": repr(exc)[:400]}
            guarded("cfg2", leg_cfg2, dev)
            if args.precision == "bf16":
                guarded("fp32", leg_fp32, dev, model, table_host, hist_idx, h_off, cand_idx, c_off, n_imp, n_c)
        hostmem.restore_affinity()  # the host-side baselines get every core again
        if not args.no_cpu_baseline:
            guarded("cpu_baseline", cpu_baseline, 4 * args.ref_sample, 1)  # ~10-30 s of host work
        if extras:
            out["reference_gpu"] = reference_gpu_subprocess()
    if rank == 0:
        print(json.dumps(out), flush=True)
    D.close()


# ------------------------------------------------------------------------------------------------
def leg_e2e(args, D, eng, model, table_host, hist_idx, h_off, cand_idx, c_off, n_imp, n_h, n_c, scores, ranks, numa):
    """Host buffers in, host buffers out, through ScoringEngine (the object behind the reference-named seams)."""
    from news_recommendation_project_v2_b200.engine import ScoringEngine

    dev = D.dev
    pin = lambda x: x.cpu().pin_memory()
    hi_h, ci_h, ho_h, co_h = pin(hist_idx), pin(cand_idx), pin(h_off), pin(c_off)
    scores_h = torch.empty(n_c, dtype=torch.float32).pin_memory()
    ranks_h = torch.empty(n_c, dtype=torch.int16).pin_memory()  # dense ranks <= 300 here: 2 bytes on the wire
    idx_bytes = (n_h + n_c) * 4 + 2 * (n_imp + 1) * 8
    table_bytes = table_host.numel() * 4
    d2h = n_c * (4 + 2)
    t0, t1 = _ev(), _ev()

    def cold_step():
        # public host API: streamed table upload + row transform, then chunk-pipelined H2D | score | D2H
        e = ScoringEngine(table_host, model, precision=args.precision, device=dev, cache_table=False)
        e.score_host(hi_h, ho_h, ci_h, co_h, scores_out=scores_h, ranks_out=ranks_h, n_chunks=E2E_CHUNKS)

    def warm_step():
        # engine resident (cached_engine semantics: same table object, same weights): the row transform is redone
        # like in the resident `value` step; this step's indices go in and its scores / ranks come out
        eng.prepare_user_encoder(eng.cand)
        eng.score_host(hi_h, ho_h, ci_h, co_h, scores_out=scores_h, ranks_out=ranks_h, n_chunks=E2E_CHUNKS)

    res = {}
    e_steps = max(2, min(args.steps, 5))
    for name, fn in (("cold", cold_step), ("warm", warm_step)):
        for _ in range(2):
            fn()
        D.barrier()
        t0.record()
        for _ in range(e_steps):
            fn()
        t1.record()
        D.barrier()
        ms = D.max_ms(t0.elapsed_time(t1)) / e_steps
        res[name] = (n_imp * D.world / (ms * 1e-3), ms)
        assert torch.equal(scores_h, scores.cpu()) and torch.equal(ranks_h.to(torch.int32), ranks.cpu()), \
            "e2e and resident paths differ"
    # what the links deliver with every rank copying at once (names the multi-GPU limiter from numbers)
    probe = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    probe_d = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    bw = {}
    for name, (dst, src) in (("h2d", (probe_d, probe)), ("d2h", (probe, probe_d))):
        dst.copy_(src, non_blocking=True)
        D.barrier()
        t0.record()
        for _ in range(4):
            dst.copy_(src, non_blocking=True)
        t1.record()
        D.barrier()
        per_rank = D.gather_floats(4 * probe.numel() / (t0.elapsed_time(t1) * 1e-3) / 1e9)
        bw[name + "_gbs_per_rank_all_ranks_copying"] = [round(v, 1) for v in per_rank]
    cold_v, cold_ms = res["cold"]
    warm_v, warm_ms = res["warm"]
    # headline e2e = the call a user of the public API makes repeatedly: `cached_engine` keeps the engine (table,
    # transformed tables, kernel-ready weights) resident while the table object and the weights are unchanged -- every
    # epoch of the reference's trainers and every further eval.py pass hit that path -- and EVERY step still copies
    # its own inputs (CSR indices) in and its results (scores, ranks) out.  `cold` = a first call on a new table.
    return {"value": round(warm_v, 1), "unit": UNIT, "h2d_bytes_per_step": int(idx_bytes),
            "d2h_bytes_per_step": int(d2h), "steps": e_steps, "ms_per_step": round(warm_ms, 3),
            "achieved_h2d_gbs_per_rank": round(idx_bytes / (warm_ms * 1e-3) / 1e9, 2),
            "achieved_d2h_gbs_per_rank": round(d2h / (warm_ms * 1e-3) / 1e9, 2),
            "what": "engine resident across steps (cached_engine semantics: same table object and weights); the per-row "
                    "transform still runs every step; this step's CSR indices are copied in from pinned host memory and "
                    "its scores (fp32) / ranks (int16) are copied out, chunk-pipelined H2D | kernel | D2H (the index copies start "
                    "while the transform still runs: engine-owned device staging, chunk plan by bisection)",
            "cold": {"value": round(cold_v, 1), "ms_per_step": round(cold_ms, 3),
                     "h2d_bytes_per_step": int(table_bytes + idx_bytes), "d2h_bytes_per_step": int(d2h),
                     "what": "a NEW engine every step: the pinned fp32 table (0.66 GB) is uploaded, rounded to bf16 and "
                             "transformed again before the first impression can be scored"},
            "link_probe": bw, "host_numa": numa,
            "e2e_check": "scores (fp32) and ranks (int16 on the wire) of both e2e flavours are bit-identical to the "
                         "resident step's"}


# ------------------------------------------------------------------------------------------------
def leg_strong(args, D, model, eng_weak, weak_ms_step, peaks):
    """BASELINE configs[3] as written: 2.4 M impressions TOTAL, impression-sharded over the ranks.  The raw table
    is replicated; its per-row transform is partitioned (each rank transforms rows [g*N/W, (g+1)*N/W) and the
    transformed rows are all-gathered by the copy engines over NVLink); each rank scores its cost-balanced block."""
    from news_recommendation_project_v2_b200 import _lib, ops
    from news_recommendation_project_v2_b200.sharded import ShardedTableEngine
    from news_recommendation_project_v2_b200.sharding import partition_impressions, table_shard_bounds

    dev, rank, world = D.dev, D.rank, D.world
    lib = _lib.load()
    n_total = 2_400_000
    hist_idx, h_off, cand_idx, c_off, hist_len, cand_len, n_h, n_c = make_device_impressions(
        n_total, N_ROWS, H_MAX, 1234, dev)  # the same global set on every rank
    a, b = partition_impressions(hist_len.cpu().numpy(), cand_len.cpu().numpy(), world)[rank]
    ho, co = h_off[a:b + 1].contiguous(), c_off[a:b + 1].contiguous()
    my_c = int(co[-1] - co[0])
    my_h = int(ho[-1] - ho[0])
    table = eng_weak.cand  # replicated raw table, engine dtype, already resident
    r0, r1 = table_shard_bounds(N_ROWS, world)[rank]
    chunk = max(256, -(-(r1 - r0) // max(1, args.strong_chunks)))
    eng = ShardedTableEngine(table[r0:r1], N_ROWS, model, precision=args.precision, device=dev, gather=args.gather
                             if args.gather != "none" else "auto", chunk_rows=chunk, cand_table=table)
    scores = torch.empty(n_c, dtype=torch.float32, device=dev)
    ranks = torch.empty(n_c, dtype=torch.int32, device=dev)
    flag = ops.new_err_flag(dev)

    def step(evs=None):
        if evs:
            evs[0].record()
        eng.build(table[r0:r1])
        if evs:
            evs[1].record()
        eng.score_device(hist_idx, ho, cand_idx, co, n_c, want_ranks=True, err_flag=flag, out_scores=scores,
                         out_ranks=ranks)
        if evs:
            evs[2].record()

    for _ in range(3):
        step()
    D.barrier()
    steps = max(args.steps, 5)
    kev = [(_ev(), _ev(), _ev()) for _ in range(steps)]
    t0, t1 = _ev(), _ev()
    l0 = lib.nrb_kernel_launches()
    t0.record()
    for i in range(steps):
        step(kev[i])
    t1.record()
    D.barrier()
    launches = lib.nrb_kernel_launches() - l0
    ops.raise_on_index_error(flag, "bench strong")
    ms = D.max_ms(t0.elapsed_time(t1)) / steps
    build_ms = float(np.mean([x.elapsed_time(y) for x, y, _ in kev]))
    score_ms = float(np.mean([y.elapsed_time(z) for _, y, z in kev]))
    # the sharded build must give the very tables the replicated engine holds
    same = bool(torch.equal(eng.hist_x, eng_weak.hist_x) and torch.equal(eng.hist_e, eng_weak.hist_e))
    es = 2 if args.precision == "bf16" else 4
    alg = (2 * my_h + my_c) * DIM * es + 4 * (my_h + my_c) + 8 * my_c
    res = {"impressions_total": n_total, "value": round(n_total / (ms * 1e-3), 1), "unit": UNIT,
           "ms_per_step": round(ms, 3), "steps": steps, "scaling": "strong",
           "speedup_vs_single_gpu_step": round(weak_ms_step * n_total / args.impressions / ms, 3),
           "efficiency": round(weak_ms_step * n_total / args.impressions / ms / world, 4),
           "single_gpu_step_ms": round(weak_ms_step * n_total / args.impressions, 3),
           "rank_build_ms": [round(v, 3) for v in D.gather_floats(build_ms)],
           "rank_score_ms": [round(v, 3) for v in D.gather_floats(score_ms)],
           "rank0_score_gbs": round(alg / (score_ms * 1e-3) / 1e9, 1),
           "rows_transformed_per_rank": r1 - r0, "chunks_per_rank": -(-(r1 - r0) // chunk),
           "allgather_bytes_in_per_gpu": int(2 * (N_ROWS - (r1 - r0)) * DIM * es),
           "gather": eng.gather, "gpu_launches": int(launches),
           "sharded_tables_equal_replicated": same,
           "what": "step = transform own row shard (5 tcgen05 GEMMs) + copy-engine all-gather of the transformed rows "
                   "over NVLink, bracketed by two 4-byte NCCL all-reduces as stream barriers + fused score/rank of "
                   "this rank's impression block; single_gpu_step_ms = this run's own per-rank weak step (the same "
                   "2.4 M-impression work on one GPU)"}
    del eng
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------
def leg_cfg5(args, D, peaks, standalone: bool = False):
    """BASELINE configs[4]: history <= 200, d=1024, 1024 latents (latent-attention user encoder), table
    row-sharded over the ranks: step = per-shard row transform + all-gather over NVLink + local scoring."""
    from news_recommendation_project_v2_b200 import _lib, ops
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    from news_recommendation_project_v2_b200.sharded import ShardedTableEngine
    from news_recommendation_project_v2_b200.sharding import table_shard_bounds

    dev, rank, world = D.dev, D.rank, D.world
    lib = _lib.load()
    d, L, h_max = 1024, 1024, 200
    n_rows = args.table_rows if args.table_rows > 0 else 1_250_000 * world
    chunk_rows = args.chunk_rows if args.chunk_rows > 0 else int(os.environ.get("NRB200_CFG5_CHUNK_ROWS", "32768"))
    n_imp = max(1, 1_048_576 // world) if (args.impressions == 2_400_000 or not standalone) else args.impressions
    model = LatentAttentionModel(dim=d, num_latents=L, precision="bf16").eval()
    model.load_state_dict(syn.make_latent_state_dict(d, L, seed=1234))
    model.to(dev)
    r0, r1 = table_shard_bounds(n_rows, world)[rank]
    g = torch.Generator(device=dev).manual_seed(4321 + rank)
    local_rows = torch.empty(r1 - r0, d, dtype=torch.bfloat16, device=dev)
    for c0 in range(0, r1 - r0, 262144):  # generated in slabs: no 5 GB fp32 temporary
        c1 = min(r1 - r0, c0 + 262144)
        local_rows[c0:c1] = torch.nn.functional.normalize(
            torch.randn(c1 - c0, d, generator=g, device=dev, dtype=torch.float32), dim=-1).to(torch.bfloat16)
    hist_idx, h_off, cand_idx, c_off, _, _, n_h, n_c = make_device_impressions(n_imp, n_rows, h_max, 1234 + rank, dev)
    eng = ShardedTableEngine(local_rows, n_rows, model, precision="bf16", device=dev, gather=args.gather,
                             chunk_rows=chunk_rows)
    scores = torch.empty(n_c, dtype=torch.float32, device=dev)
    ranks = torch.empty(n_c, dtype=torch.int32, device=dev)
    flag = ops.new_err_flag(dev)

    def step(evs=None):
        if evs:
            evs[0].record()
        eng.build(local_rows)
        if evs:
            evs[1].record()
        eng.score_device(hist_idx, h_off, cand_idx, c_off, n_c, want_ranks=True, err_flag=flag, out_scores=scores,
                         out_ranks=ranks)
        if evs:
            evs[2].record()

    steps = args.steps if standalone else 3
    for _ in range(max(args.warmup, 1) if standalone else 1):
        step()
    D.barrier()
    launches0 = lib.nrb_kernel_launches()
    kev = [(_ev(), _ev(), _ev()) for _ in range(steps)]
    t0, t1 = _ev(), _ev()
    sampler = ClockSampler(D.local)
    if rank == 0:
        sampler.start()
    t0.record()
    for i in range(steps):
        step(kev[i])
    t1.record()
    D.barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = lib.nrb_kernel_launches() - launches0
    ops.raise_on_index_error(flag, "bench cfg5")
    if standalone and args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, scores, ranks, c_off)
    ms_step = D.max_ms(t0.elapsed_time(t1)) / steps
    build_ms = float(np.mean([a.elapsed_time(b) for a, b, _ in kev]))
    score_ms = float(np.mean([b.elapsed_time(c) for _, b, c in kev]))

    # ---- sharded == locally recomputed, bit for bit, on a sample of PEER-owned rows -----------------
    identical = None
    if eng.gather != "none":
        peer = (rank + 1) % world
        p0, p1 = table_shard_bounds(n_rows, world)[peer]
        gs = torch.Generator(device=dev).manual_seed(99 + rank)
        pick = (p0 + torch.randint(0, p1 - p0, (1024,), generator=gs, device=dev)).sort().values
        raw = eng.cand[pick].contiguous()  # rows that came over NVLink
        fw = model.folded(torch.bfloat16, dev)
        again = ops.latent_forward(fw, raw.view(-1, 1, d), None, max_tokens=65536).view(-1, d)
        again_bf = ops.convert_rows(again, torch.bfloat16)
        identical = bool(torch.equal(again_bf, eng.hist_x[pick]))
        ok = torch.tensor([1.0 if identical else 0.0], dtype=torch.float64, device=dev)
        if world > 1:
            D.dist.all_reduce(ok, op=D.dist.ReduceOp.MIN)
        identical = bool(ok.item() == 1.0)

    f_row = 4 * 8 * d * L + 24 * d * d  # executed FLOPs per row (folded heads)
    f_row_ref = 4 * d * 4096 + 4 * 4096 * L + 24 * d * d
    alg_bytes = (n_h + n_c) * d * 2 + 4 * (n_h + n_c) + 8 * n_c
    bytes_out = 2 * (r1 - r0) * d * 2 * (world - 1)
    bytes_in = 2 * (n_rows - (r1 - r0)) * d * 2
    tf_exec = (r1 - r0) * f_row / (build_ms * 1e-3) / 1e12
    res = {
        "metric": METRIC, "value": round(n_imp * world / (ms_step * 1e-3), 1), "unit": UNIT, "n_gpus": world,
        "steps": steps, "warmup": max(args.warmup, 1) if standalone else 1, "ms_per_step": round(ms_step, 3),
        "higher_is_better": True, "scaling": "weak" if args.table_rows <= 0 else "strong", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "long-history stress (BASELINE configs[4]): latent-attention user encoder, table "
                               "row-sharded, per-shard transform + all-gather (%s) + gather/pool/cosine/rank" % eng.gather,
                   "table_rows": n_rows, "rows_per_gpu": r1 - r0, "impressions_per_gpu": n_imp, "dim": d, "latents": L,
                   "history_max": h_max, "sum_history": n_h, "sum_candidates": n_c, "chunk_rows": chunk_rows},
        "gpu_launches": int(launches),
        "build": {"ms": round(build_ms, 3), "rank_ms": [round(v, 3) for v in D.gather_floats(build_ms)],
                  "tflops_executed": round(tf_exec, 1),
                  "frac_of_sustained_peak_executed": round(tf_exec / peaks["bf16_tflops_sustained"], 4),
                  "tflops_reference_formulation": round((r1 - r0) * f_row_ref / (build_ms * 1e-3) / 1e12, 1),
                  "allgather_bytes_in_per_gpu": int(bytes_in), "allgather_bytes_out_per_gpu": int(bytes_out),
                  "allgather_gbs_in_per_gpu": round(bytes_in / (build_ms * 1e-3) / 1e9, 1),
                  "allgather_gbs_out_per_gpu": round(bytes_out / (build_ms * 1e-3) / 1e9, 1),
                  "note": "the all-gather overlaps the transform chunk by chunk: GB/s = bytes / whole build time"},
        "sharded_equals_local_recompute_on_peer_rows": identical,
        "roofline": {"bound": "hbm", "kernel": "score_rank_kernel", "achieved": round(alg_bytes / (score_ms * 1e-3) / 1e9, 1),
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(alg_bytes / (score_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                     "traffic": None, "kernel_ms": round(score_ms, 3)},
        "clocks": clocks,
    }
    del eng
    torch.cuda.empty_cache()
    return res


def run_sharded(args):
    from news_recommendation_project_v2_b200 import _lib

    _stdout_to_stderr_for_native_libs()
    D = Dist(need_group=True)
    _lib.require_device(D.dev)
    res = leg_cfg5(args, D, measured_peaks(), standalone=True)
    if D.rank == 0:
        print(json.dumps(res), flush=True)
    D.close()


# ------------------------------------------------------------------------------------------------
def _stage_a_model(dev, d=768, L=512):
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel

    m = LatentAttentionModel(dim=d, num_latents=L, precision="bf16").eval()
    m.load_state_dict(syn.make_latent_state_dict(d, L, seed=1234))
    return m.to(dev)


def _stage_a_flops(d, L, heads=8, dim_head=512):
    inner = heads * dim_head
    f_ref = 4 * d * inner + 4 * inner * L + 24 * d * d  # reference formulation, K/V projection excluded
    f_exec = 4 * heads * d * L + 24 * d * d  # executed (Wq.K^T and V.Wout folded)
    return f_ref, f_exec


def _stage_a_batch(items, S, d, gen, dev):
    x = torch.randn(items, S, d, generator=gen, device=dev, dtype=torch.bfloat16)
    lens = torch.randint(8, S + 1, (items,), generator=gen, device=dev)
    mask = (torch.arange(S, device=dev)[None, :] < lens[:, None]).to(torch.int32)
    return x, mask


def bench_stage_a(dev, peaks, args):
    """configs[2] shape (seq 64, d 768, 512 latents, bf16): a 32,768-item chunk of the 1M-item job."""
    from news_recommendation_project_v2_b200 import _lib, config as nrb_config

    d, L, S, items = 768, 512, 64, 32768
    m = _stage_a_model(dev, d, L)
    g = torch.Generator(device=dev).manual_seed(1234)
    x, mask = _stage_a_batch(items, S, d, g, dev)
    valid = int(mask.sum())
    old = nrb_config.LATENT_MAX_TOKENS
    nrb_config.LATENT_MAX_TOKENS = int(os.environ.get("NRB200_BENCH_STAGE_A_TOKENS", str(old)))
    lib = _lib.load()
    try:
        for _ in range(2):
            out = m(x, mask)
        torch.cuda.synchronize()
        t0, t1 = _ev(), _ev()
        reps = 5
        l0 = lib.nrb_kernel_launches()
        t0.record()
        for _ in range(reps):
            out = m(x, mask)
        t1.record()
        torch.cuda.synchronize()
        launches = (lib.nrb_kernel_launches() - l0) / reps
    finally:
        nrb_config.LATENT_MAX_TOKENS = old
    ms = t0.elapsed_time(t1) / reps
    f_ref, f_exec = _stage_a_flops(d, L)
    tf_ref = valid * f_ref / (ms * 1e-3) / 1e12
    tf_exec = valid * f_exec / (ms * 1e-3) / 1e12
    return {"workload": "latent-attention pooling, %d items x %d tokens, d=%d, L=%d, bf16 (BASELINE configs[2] chunk)"
                        % (items, S, d, L),
            "news_per_s": round(items / (ms * 1e-3), 1), "valid_tokens": valid, "ms": round(ms, 3),
            "kernel_launches_per_call": launches,
            "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": peaks["bf16_tflops_sustained"],
                         "achieved_reference_flops": round(tf_ref, 1), "achieved_executed_flops": round(tf_exec, 1),
                         "frac": round(tf_ref / peaks["bf16_tflops_sustained"], 4),
                         "frac_executed": round(tf_exec / peaks["bf16_tflops_sustained"], 4),
                         "peak_source": peaks["source"]},
            "finite": bool(torch.isfinite(out).all())}


def leg_cfg3(dev, peaks):
    """BASELINE configs[2] in full: 1,000,000 synthetic news items (seq 64, d 768, 512 latents, bf16) through the
    fused latent-attention pooling on one GPU, streamed in 65,536-item chunks generated on the device (the padded
    input would be 98 GB).  Timed: the pooling calls only (CUDA events per chunk); generating a chunk is not."""
    d, L, S, total, chunk = 768, 512, 64, 1_000_000, 65_536
    m = _stage_a_model(dev, d, L)
    g = torch.Generator(device=dev).manual_seed(4242)
    x, mask = _stage_a_batch(4096, S, d, g, dev)
    m(x, mask)  # warm-up (weights folded, workspace sized)
    ms_sum, valid, n_done, finite = 0.0, 0, 0, True
    unit_norm_err = 0.0
    t0, t1 = _ev(), _ev()
    while n_done < total:
        items = min(chunk, total - n_done)
        x, mask = _stage_a_batch(items, S, d, g, dev)
        torch.cuda.synchronize()
        t0.record()
        out = m(x, mask)
        t1.record()
        torch.cuda.synchronize()
        ms_sum += t0.elapsed_time(t1)
        valid += int(mask.sum())
        finite = finite and bool(torch.isfinite(out).all())
        unit_norm_err = max(unit_norm_err, float((out.norm(dim=-1) - 1).abs().max()))
        n_done += items
        del x, mask, out
    f_ref, f_exec = _stage_a_flops(d, L)
    tf_ref = valid * f_ref / (ms_sum * 1e-3) / 1e12
    tf_exec = valid * f_exec / (ms_sum * 1e-3) / 1e12
    return {"workload": "save_emb-style bulk news encoding (BASELINE configs[2]): %d items x %d tokens, d=%d, L=%d, "
                        "bf16, %d-item chunks generated on device" % (total, S, d, L, chunk),
            "news_per_s": round(total / (ms_sum * 1e-3), 1), "seconds": round(ms_sum * 1e-3, 3),
            "valid_tokens": valid, "tokens_per_s": round(valid / (ms_sum * 1e-3), 1),
            "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": peaks["bf16_tflops_sustained"],
                         "achieved_reference_flops": round(tf_ref, 1), "achieved_executed_flops": round(tf_exec, 1),
                         "frac": round(tf_ref / peaks["bf16_tflops_sustained"], 4),
                         "frac_executed": round(tf_exec / peaks["bf16_tflops_sustained"], 4)},
            "finite": finite, "max_unit_norm_err": unit_norm_err}


def leg_cfg3_e2e(dev):
    """Stage A end to end from the packed token FILE (the format in front of stage A): page cache -> pinned staging
    (parallel memcpy) -> H2D -> varlen latent-attention pooling -> D2H, double buffered, on a bounded 65,536-item
    sample of the cfg-3 workload (the full job's tokens are 55 GB)."""
    import shutil
    import tempfile

    from news_recommendation_project_v2_b200.token_store import (PackedTokenFile, apply_token_attn_packed,
                                                                 write_packed_tokens)

    d, L, S, items, slab = 768, 512, 64, 65_536, 4096
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > (12 << 30) \
        else tempfile.gettempdir()
    path = os.path.join(base, "nrb200_cfg3_%d.nrbtok" % os.getpid())
    m = _stage_a_model(dev, d, L)

    def gen():
        g = torch.Generator(device=dev).manual_seed(777)
        for _ in range(0, items, slab):
            x, mask = _stage_a_batch(slab, S, d, g, dev)
            lens = mask.sum(1).cpu().tolist()
            xc = x.cpu()
            for i in range(slab):
                yield xc[i, :lens[i]]

    try:
        n_items, n_tok = write_packed_tokens(path, gen(), d)
        tf = PackedTokenFile(path)
        threads = max(1, min(16, (os.cpu_count() or 2) - 1))
        timings = {}
        reg_s = None
        for mode in ("staged", "registered"):
            if mode == "registered":
                t = time.perf_counter()
                ok = tf.tokens_raw.nbytes <= (8 << 30) and tf.register()  # page-locking costs seconds per GB, once
                reg_s = time.perf_counter() - t
                if not ok:
                    timings[mode] = None
                    continue
            out = apply_token_attn_packed(m, tf, copy_threads=threads)  # warm-up: page cache, workspace, pinned pools
            torch.cuda.synchronize()
            t = time.perf_counter()
            reps = 2
            for _ in range(reps):
                out = apply_token_attn_packed(m, tf, copy_threads=threads, out=out)
            timings[mode] = (time.perf_counter() - t) / reps
        tf.unregister()
        dt = min(v for v in timings.values() if v)
    finally:
        if os.path.exists(path):
            os.remove(path)
    h2d = n_tok * d * 2
    return {"value": round(n_items / dt, 1), "unit": "news/s", "seconds": round(dt, 4), "items": n_items,
            "valid_tokens": n_tok, "h2d_bytes_per_pass": int(h2d), "d2h_bytes_per_pass": int(n_items * d * 4),
            "achieved_h2d_gbs": round(h2d / dt / 1e9, 2), "copy_threads": threads, "file_on": base,
            "seconds_staged_through_pinned_buffers": round(timings["staged"], 4),
            "seconds_mapping_page_locked": None if timings["registered"] is None else round(timings["registered"], 4),
            "seconds_page_locking_the_mapping_once": None if reg_s is None else round(reg_s, 2),
            "register_attempts": getattr(tf, "register_error", None),
            "finite": bool(torch.isfinite(out).all()),
            "max_unit_norm_err": float((out.norm(dim=-1) - 1).abs().max()),
            "what": "packed token file (mmap, page cache) -> H2D -> nrb_latent_forward_packed -> D2H of the pooled "
                    "vectors, wall clock of a whole pass; `value` = the faster of two modes: staged through pinned double "
                    "buffers (parallel memcpy, no set-up), or DMA straight from the page-locked mapping (cudaHostRegister "
                    "of the shared mapping once -- seconds per GB -- which pays when the store is read again, e.g. every "
                    "epoch)"}


def _time_calls(fn, reps):
    t0, t1 = _ev(), _ev()
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps * 1e3  # us


def _graph_us(fn, reps):
    """The same launches captured once in a CUDA graph and replayed (launch-bound inner loop)."""
    try:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                fn()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        from news_recommendation_project_v2_b200 import ops

        before = set(ops._ws_cache)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        us = round(_time_calls(g.replay, reps), 2)
        for k in set(ops._ws_cache) - before:  # scratch taken from the graph's private pool dies with the graph
            ops._ws_cache.pop(k, None)
        return us, None
    except Exception as e:  # pragma: no cover - reported, not hidden
        torch.cuda.synchronize()
        return None, repr(e)[:200]


def leg_cfg2(dev):
    """BASELINE configs[1]: the configs[0] model on one B200 at batch 1,024 impressions, bf16 -- about 60 MB of row
    reads, i.e. ~10 us of HBM time: launch-latency bound, so it is reported as latency (eager and graph replay)."""
    from news_recommendation_project_v2_b200 import ops
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention

    d, n_rows, n_imp, S, L = 768, 65_536, 1024, 64, 512
    fa = FinalAttention(d, HIDDEN, precision="bf16").eval()
    fa.load_state_dict(syn.make_final_attention_state_dict(d, HIDDEN, seed=1234))
    table = syn.make_table(n_rows, d, seed=1234)
    eng = ScoringEngine(table, fa.to(dev), precision="bf16", device=dev)
    hi, ho, ci, co, hl, cl, n_h, n_c = make_device_impressions(n_imp, n_rows, H_MAX, 77, dev, cand="small")
    scores = torch.empty(n_c, dtype=torch.float32, device=dev)
    ranks = torch.empty(n_c, dtype=torch.int32, device=dev)
    flag = ops.new_err_flag(dev)
    score = lambda: eng.score_device(hi, ho, ci, co, n_c, want_ranks=True, err_flag=flag, out_scores=scores,
                                     out_ranks=ranks)
    score_us = _time_calls(score, 200)
    score_graph_us, gerr = _graph_us(score, 200)
    alg = (2 * n_h + n_c) * d * 2 + 4 * (n_h + n_c) + 8 * n_c
    # host API, engine cached: numpy index arrays in, numpy scores + rank arrays out (includes H2D, D2H, sync)
    hi_n, hl_n, ci_n, cl_n = hi.cpu().numpy(), hl.cpu().numpy(), ci.cpu().numpy(), cl.cpu().numpy()

    def host_call():
        _, s, r = eng.score(hi_n, hl_n, ci_n, cl_n)
        return s.cpu(), r.cpu()

    for _ in range(3):
        host_call()
    t = time.perf_counter()
    for _ in range(50):
        host_call()
    host_us = (time.perf_counter() - t) / 50 * 1e6
    # stage A on the batch: 1,024 news items x 64 tokens through the latent-attention pooling
    m = _stage_a_model(dev, d, L)
    g = torch.Generator(device=dev).manual_seed(5)
    x, mask = _stage_a_batch(n_imp, S, d, g, dev)
    pool = lambda: m(x, mask)
    pool_us = _time_calls(pool, 50)
    pool_graph_us, gerr2 = _graph_us(pool, 50)
    valid = int(mask.sum())
    _, f_exec = _stage_a_flops(d, L)
    res = {"workload": "BASELINE configs[1]: 1,024 impressions (H<=50, C in [3,7]), d=768, N=65,536, bf16; "
                       "1,024 news items x 64 tokens for stage A",
           "score_rank_us": round(score_us, 2), "score_rank_graph_us": score_graph_us,
           "score_rank_impressions_per_s": round(n_imp / (score_us * 1e-6), 1),
           "score_rank_algorithmic_gbs": round(alg / (score_us * 1e-6) / 1e9, 1),
           "host_api_us": round(host_us, 1), "host_api_impressions_per_s": round(n_imp / (host_us * 1e-6), 1),
           "stage_a_us": round(pool_us, 1), "stage_a_graph_us": pool_graph_us,
           "stage_a_news_per_s": round(n_imp / (pool_us * 1e-6), 1),
           "stage_a_tflops_executed": round(valid * f_exec / (pool_us * 1e-6) / 1e12, 1)}
    if gerr or gerr2:
        res["graph_error"] = gerr or gerr2
    return res


def leg_fp32(dev, model_bf16, table_host, hist_idx, h_off, cand_idx, c_off, n_imp, n_c):
    """The rank-exact path (fp32 tables) on the headline workload, the number that goes with the bit-exact-rank
    evidence of tests/test_gpu_api.py: "fp32" = FFMA row transform (the reference's own arithmetic); "fp32x3" = the
    same tables with the row transform on the tensor cores as split-bf16 GEMMs (hi/lo operand pairs, three products
    accumulated in fp32), held to the same 1e-5 score bar by the same tests."""
    from news_recommendation_project_v2_b200 import ops
    from news_recommendation_project_v2_b200.engine import ScoringEngine
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention

    n_h = int(h_off[-1])
    alg = (2 * n_h + n_c) * DIM * 4 + 4 * (n_h + n_c) + 8 * n_c
    res, ref_scores = {}, None
    for precision in ("fp32", "fp32x3"):
        m32 = FinalAttention(DIM, HIDDEN, precision=precision).eval()
        m32.load_state_dict(model_bf16.state_dict())
        eng = ScoringEngine(table_host, m32.to(dev), precision=precision, device=dev)
        scores = torch.empty(n_c, dtype=torch.float32, device=dev)
        ranks = torch.empty(n_c, dtype=torch.int32, device=dev)
        flag = ops.new_err_flag(dev)
        evs = [(_ev(), _ev(), _ev()) for _ in range(3)]

        def step(e=None):
            if e:
                e[0].record()
            eng.prepare_user_encoder(eng.cand)
            if e:
                e[1].record()
            eng.score_device(hist_idx, h_off, cand_idx, c_off, n_c, want_ranks=True, err_flag=flag, out_scores=scores,
                             out_ranks=ranks)
            if e:
                e[2].record()

        step()
        torch.cuda.synchronize()
        for e in evs:
            step(e)
        torch.cuda.synchronize()
        tr = float(np.mean([a.elapsed_time(b) for a, b, _ in evs]))
        sc = float(np.mean([b.elapsed_time(c) for _, b, c in evs]))
        r = {"value": round(n_imp / ((tr + sc) * 1e-3), 1), "unit": UNIT, "ms_per_step": round(tr + sc, 3),
             "row_transform_ms": round(tr, 3), "score_rank_ms": round(sc, 3),
             "score_rank_gbs": round(alg / (sc * 1e-3) / 1e9, 1)}
        if precision == "fp32":
            r["row_transform_tflops_ffma"] = round(N_ROWS * 67.1e6 / (tr * 1e-3) / 1e12, 1)
            ref_scores, ref_ranks = scores.clone(), ranks.clone()
            res.update(r)
            res["what"] = ("fp32 tables + FFMA (gemm_simt) transform: scores within 1e-5 of the reference, ranks "
                           "bit-exact wherever the reference's score gaps exceed that (test_gpu_api.py)")
        else:
            r["row_transform_tflops_tensor_executed"] = round(3 * N_ROWS * 67.1e6 / (tr * 1e-3) / 1e12, 1)
            r["max_abs_score_diff_vs_fp32"] = float((scores - ref_scores).abs().max())
            r["impressions_with_rank_diff_vs_fp32"] = int(torch.unique(torch.bucketize(
                torch.nonzero(ranks != ref_ranks).flatten(), c_off[1:], right=True)).numel())
            r["what"] = ("fp32 tables, row transform as split-bf16 tcgen05 GEMMs (K' = 3K: a_hi w_hi + a_hi w_lo + "
                         "a_lo w_hi accumulated in fp32)")
            res["fp32x3"] = r
        del eng
        torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------
def _reference_step_fn(device: str, batch_size: int):
    """A callable running the reference's own get_final_second_attention_score on (sd, table, impressions), and
    what it is: the UNMODIFIED reference (oracle/_ref or /root/reference) when present, else the oracle port."""
    from oracle import ref_harness  # the reference arm / cpu_baseline legs are where bench may run oracle/

    if ref_harness.reference_available():
        import pandas as pd

        ref = ref_harness.load_reference(batch_size=batch_size, device=device)
        model = ref_harness.make_reference_final_attention(ref, DIM, HIDDEN, seed=1234)
        model.load_state_dict(syn.make_final_attention_state_dict(DIM, HIDDEN, seed=1234))
        model = model.to(device).eval()

        def run(table, imp):
            hb = pd.Series(np.ones(imp.n, dtype=bool))
            with torch.no_grad():
                return ref.data_model_helper.get_final_second_attention_score(
                    imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, hb, model)

        return run, "reference", ("the unmodified reference: news_rec_utils.data_model_helper."
                                  "get_final_second_attention_score from %s" % ref_harness.reference_origin())
    from oracle import oracle

    sd = syn.make_final_attention_state_dict(DIM, HIDDEN, seed=1234)

    def run_port(table, imp):
        return oracle.final_second_attention_score(sd, table, imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len,
                                                   dtype=torch.float32, batch=batch_size)

    return run_port, "port", "oracle port of the reference path (oracle/_ref not installed)"


def _quiet(fn, *a):
    """The reference prints progress bars / messages on stdout; keep stdout to the JSON line."""
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        return fn(*a)


def cpu_baseline(sample: int, steps: int):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    run, kind, what = _reference_step_fn("cpu", 64)
    table = syn.make_table(N_ROWS, DIM, seed=1234)
    imp = syn.make_impressions(sample, N_ROWS, h_max=H_MAX, cand="large", seed=1234)
    _quiet(run, table, syn.make_impressions(64, N_ROWS, h_max=H_MAX, cand="large", seed=1))  # thread pool warm-up
    t = time.perf_counter()
    for _ in range(steps):
        _quiet(run, table, imp)
    dt = (time.perf_counter() - t) / steps
    return {"value": round(sample / dt, 2), "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "%d cfg-4-shaped impressions (d=%d, H<=%d, C~37), fp32 torch CPU ops; %s (per-slot "
                      "FinalAttention MLP + per-impression cosine + scipy dense rank)" % (sample, DIM, H_MAX, what)}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation (the unmodified package installed into oracle/_ref by
    oracle/build_ref.py; the oracle port only if that is missing) on the host cores, same metric/config, each
    step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["CUDA_VISIBLE_DEVICES"] = ""  # the CPU arm: the reference's DEVICE constant then resolves to cpu
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    run, kind, what = _reference_step_fn("cpu", 64)
    table = syn.make_table(N_ROWS, DIM, seed=1234)
    imp = syn.make_impressions(args.ref_sample, N_ROWS, h_max=H_MAX, cand="large", seed=1234)
    for _ in range(args.warmup):
        _quiet(run, table, imp)
    t = time.perf_counter()
    for _ in range(args.steps):
        _quiet(run, table, imp)
    dt = (time.perf_counter() - t) / args.steps
    value = args.ref_sample / dt
    sample = ("%d cfg-4-shaped impressions per step (d=%d, H<=%d, C~37), fp32, %s, %d threads"
              % (args.ref_sample, DIM, H_MAX, what, cores))
    out = {
        "impl": "reference", "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "table_rows": N_ROWS, "dim": DIM, "hidden": HIDDEN,
                   "history_max": H_MAX, "impressions_per_step": args.ref_sample},
        "cpu_baseline": {"value": round(value, 2), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": round(value, 2), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def run_reference_gpu(args):
    """The same reference code with DEVICE=cuda (config.py:19) on this box's GPU: CPU gather in the DataLoader
    collate, per-batch H2D, per-impression cosine loop with 2 H2D + 1 D2H each, scipy dense rank on the host."""
    _stdout_to_stderr_for_native_libs()
    from oracle import ref_harness

    if not ref_harness.reference_available():
        print(json.dumps({"impl": "reference-gpu", "unavailable": "oracle/_ref not installed"}), flush=True)
        return
    run, kind, what = _reference_step_fn("cuda", 512)
    table = syn.make_table(N_ROWS, DIM, seed=1234)
    n = max(args.ref_sample, 8192)
    imp = syn.make_impressions(n, N_ROWS, h_max=H_MAX, cand="large", seed=1234)
    _quiet(run, table, syn.make_impressions(512, N_ROWS, h_max=H_MAX, cand="large", seed=1))
    torch.cuda.synchronize()
    steps = max(1, min(args.steps, 3))
    t = time.perf_counter()
    for _ in range(steps):
        _quiet(run, table, imp)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t) / steps
    stage_a = _reference_stage_a_gpu()
    cfg2 = _reference_cfg2_gpu()
    print(json.dumps({"impl": "reference-gpu", "value": round(n / dt, 1), "unit": UNIT, "ms_per_step": round(dt * 1e3, 1),
                      "stage_a": stage_a, "cfg2": cfg2,
                      "sample": "%d cfg-4-shaped impressions per step, fp32, %s with DEVICE=cuda (torch %s on %s), user-"
                                "encoder batch 512" % (n, what, torch.__version__, torch.cuda.get_device_name(0)),
                      "steps": steps}), flush=True)


def _reference_stage_a_gpu():
    """The reference's own LatentAttentionModel (latent_attention.py:134-171) with DEVICE=cuda on this GPU, cfg-2
    shape (seq 64, d 768, 512 latents), fp32 like the reference's TORCH_DTYPE and under bf16 autocast."""
    try:
        from oracle import ref_harness

        ref = ref_harness.load_reference(batch_size=512, device="cuda")
        d, L, S, B, reps = 768, 512, 64, 256, 8
        model = ref_harness.make_reference_latent_model(ref, d, L, seed=1234)
        model.load_state_dict(syn.make_latent_state_dict(d, L, seed=1234))
        model = model.to("cuda").eval()
        g = torch.Generator(device="cuda").manual_seed(1234)
        x = torch.randn(B, S, d, generator=g, device="cuda")
        lens = torch.randint(8, S + 1, (B,), generator=g, device="cuda")
        mask = (torch.arange(S, device="cuda")[None, :] < lens[:, None]).to(torch.int32)
        out = {}
        for name, ctx in (("fp32", None), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            def run():
                with torch.no_grad():
                    if ctx is None:
                        return model(x, mask)
                    with ctx:
                        return model(x, mask)
            _quiet(run)
            torch.cuda.synchronize()
            t = time.perf_counter()
            for _ in range(reps):
                _quiet(run)
            torch.cuda.synchronize()
            out[name + "_news_per_s"] = round(B * reps / (time.perf_counter() - t), 1)
        out["sample"] = "%d x %d items x %d tokens, d=%d, L=%d, reference module on cuda" % (reps, B, S, d, L)
        return out
    except Exception as exc:  # pragma: no cover - reported, not hidden
        return {"unavailable": repr(exc)[:300]}


def _reference_cfg2_gpu():
    """BASELINE configs[1] on the reference's torch path: 1,024 impressions (H<=50, C in [3,7]), d=768, N=65,536,
    FinalAttention user encoder, DEVICE=cuda, one call of get_final_second_attention_score."""
    try:
        import pandas as pd

        from oracle import ref_harness

        ref = ref_harness.load_reference(batch_size=512, device="cuda")
        d, n_rows, n_imp = 768, 65_536, 1024
        model = ref_harness.make_reference_final_attention(ref, d, HIDDEN, seed=1234)
        model.load_state_dict(syn.make_final_attention_state_dict(d, HIDDEN, seed=1234))
        model = model.to("cuda").eval()
        table = syn.make_table(n_rows, d, seed=1234)
        imp = syn.make_impressions(n_imp, n_rows, h_max=H_MAX, cand="small", seed=77)
        hb = pd.Series(np.ones(n_imp, dtype=bool))

        def run():
            with torch.no_grad():
                return ref.data_model_helper.get_final_second_attention_score(
                    imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, table, hb, model)

        _quiet(run)
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(3):
            _quiet(run)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t) / 3
        return {"ms_per_call": round(dt * 1e3, 1), "impressions_per_s": round(n_imp / dt, 1),
                "sample": "1,024 impressions, d=768, N=65,536, fp32, reference torch path with DEVICE=cuda"}
    except Exception as exc:  # pragma: no cover - reported, not hidden
        return {"unavailable": repr(exc)[:300]}


def reference_gpu_subprocess():
    """Run `bench.py --impl reference-gpu` in a fresh process (its torch / CUDA state is the reference's own)."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-gpu", "--steps", "2"],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
        if r.returncode != 0 or not lines:
            return {"unavailable": ("exit %d: " % r.returncode) + r.stderr[-300:]}
        return json.loads(lines[-1])
    except Exception as e:  # pragma: no cover
        return {"unavailable": repr(e)[:300]}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-gpu":
        run_reference_gpu(args)
    elif args.workload == "cfg5":
        run_sharded(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
