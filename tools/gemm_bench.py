"""Micro-benchmark of the tcgen05 dense row kernel (nrb_linear) on the shapes the hot path uses.

    python tools/gemm_bench.py [tag]
"""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from news_recommendation_project_v2_b200 import ops

tag = sys.argv[1] if len(sys.argv) > 1 else "default"
dev = torch.device("cuda", 0)
M = 147456
cases = [  # name, N, K, epi, out dtype, group
    ("logits+softmax (stage A GEMM1)", 4096, 768, 5, torch.bfloat16, 512),
    ("plain bf16 out, same shape", 4096, 768, 0, torch.bfloat16, 0),
    ("relu bf16 out, same shape", 4096, 768, 1, torch.bfloat16, 0),
    ("value GEMM + residual (GEMM2)", 768, 4096, 3, torch.float32, 0),
    ("plain fp32 out, same shape", 768, 4096, 0, torch.float32, 0),
    ("plain bf16 out, same shape", 768, 4096, 0, torch.bfloat16, 0),
    ("FF1 + GEGLU (GEMM3)", 6144, 768, 4, torch.bfloat16, 0),
    ("plain bf16 out, same shape", 6144, 768, 0, torch.bfloat16, 0),
    ("FF2 + residual (GEMM4)", 768, 3072, 3, torch.float32, 0),
    ("plain fp32 out, same shape", 768, 3072, 0, torch.float32, 0),
    ("plain bf16 out, same shape", 768, 3072, 0, torch.bfloat16, 0),
    ("FinalAttention linear2 (relu)", 4096, 4096, 1, torch.bfloat16, 0),
    ("cfg5 logits+softmax L=1024", 8192, 1024, 5, torch.bfloat16, 1024),
    ("cfg5 plain bf16, same shape", 8192, 1024, 0, torch.bfloat16, 0),
]
res = []
for name, N, K, epi, odt, group in cases:
    a = torch.randn(M, K, device=dev).to(torch.bfloat16)
    w = (torch.randn(N, K, device=dev) / K ** 0.5).to(torch.bfloat16)
    bias = torch.randn(N, device=dev) * 0.1 if epi in (1, 4) or (epi == 3 and K == 3072) else None
    r = torch.randn(M, N, device=dev) if epi == 3 else None
    run = lambda: ops.linear(a, w, bias, epi, r, odt, group=group, group_valid=group)
    for _ in range(3):
        run()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(10):
        run()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / 10
    tf = 2.0 * M * N * K / ms / 1e9
    res.append(dict(name=name, M=M, N=N, K=K, epi=epi, out=str(odt).split(".")[-1], ms=round(ms, 4), tflops=round(tf, 1)))
    print(res[-1], flush=True)
    del a, w, r
os.makedirs("gpurun_out", exist_ok=True)
json.dump(res, open(f"gpurun_out/gemm_bench_{tag}.json", "w"), indent=1)
