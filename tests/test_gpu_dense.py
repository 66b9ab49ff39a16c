"""GPU parity: dense row kernels (tcgen05 bf16 / FFMA fp32) and the FinalAttention row transform.

The floating-point reference for a single contraction is plain torch in fp32/fp64 on the SAME
(already rounded) operands; the row transform is checked against the CPU oracle.
"""
import math

import numpy as np
import pytest
import torch

from oracle import oracle
from news_recommendation_project_v2_b200 import synthetic as syn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from news_recommendation_project_v2_b200 import ops as _ops
    return _ops


def _ref_linear(a, w, bias, epi, res):
    y = a.double() @ w.double().T
    if bias is not None:
        y = y + bias.double()
    if epi == 1:
        y = torch.relu(y)
    elif epi == 2:
        y = torch.exp(y)
    elif epi == 3:
        y = y + res.double()
    elif epi == 4:
        y4 = y.reshape(y.shape[0], -1, 4)  # interleaved in pairs (a0,a1,g0,g1,a2,a3,g2,g3,...)
        a_, g_ = y4[:, :, 0:2].reshape(y.shape[0], -1), y4[:, :, 2:4].reshape(y.shape[0], -1)
        y = a_ * 0.5 * g_ * (1 + torch.erf(g_ / math.sqrt(2)))
    return y


SHAPES = [(128, 256, 64), (1, 256, 128), (300, 768, 1024), (1000, 4096, 768), (257, 128, 256), (129, 64, 64),
          (4099, 1024, 4096), (640, 6144, 768),
          # partial 256-wide N tiles on the CTA pair (rank 1's W half partly / entirely past N) and the single CTA
          (300, 160, 128), (513, 384, 256), (1000, 800, 512), (100, 416, 128),
          (200, 32, 64), (1000, 96, 192)]  # small-N: one partial 128-wide tile


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("epi", [0, 1, 2, 3, 4])
def test_linear_bf16_tcgen05(ops, M, N, K, epi):
    g = torch.Generator().manual_seed(M * 7 + N + K + epi)
    a = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16)
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(torch.bfloat16)
    bias = torch.randn(N, generator=g) * 0.1
    res = torch.randn(M, N, generator=g) if epi == 3 else None
    want = _ref_linear(a, w, bias, epi, res)
    for out_dtype in (torch.float32, torch.bfloat16):
        y = ops.linear(a.cuda(), w.cuda(), bias.cuda(), epi, None if res is None else res.cuda(), out_dtype)
        assert y.dtype == out_dtype and y.shape == want.shape
        tol = 2e-4 if out_dtype == torch.float32 else 1.2e-2  # fp32 accumulate / one bf16 rounding (2^-8 rel)
        torch.testing.assert_close(y.cpu().double(), want, atol=tol, rtol=tol)
    # no-bias path
    y = ops.linear(a.cuda(), w.cuda(), None, 0 if epi != 4 else 4, None, torch.float32)
    torch.testing.assert_close(y.cpu().double(), _ref_linear(a, w, None, 0 if epi != 4 else 4, None), atol=2e-4, rtol=2e-4)


def _tiles_per_unit(M, N, rows_per_unit, bn, tiles_per_unit_row, cs):
    """Tiles each persistent CTA (or cluster / CTA pair) of the tcgen05 GEMM works through, computed the way
    launch_gemm sizes its grid: ceil(M / rows) * (ceil(N / BN) / tiles per unit) units over at most SMs / cluster
    co-resident units.  Clusters of 4 are further limited by what the GPCs can hold, which only adds tiles."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    units = -(-M // rows_per_unit) * (-(-N // bn) // tiles_per_unit_row)
    return units / (sms // cs)


def _multi_tile_shape(kind):
    """(M, N, K, group, group_valid, rows per unit, BN, N tiles per unit, cluster) with >= 3 tiles per unit; the
    last tile of some unit is partial in M and in N."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if kind == "small_n":  # BN 128 (N <= 128), one CTA per unit
        return 3 * sms * 128 - 50, 96, 192, 0, 0, 128, 128, 1, 1
    if kind == "single":  # BN 256 on one CTA: M <= 128 keeps the CTA pair out
        return 100, 3 * sms * 256 + 96, 128, 0, 0, 128, 256, 1, 1
    if kind == "pair":  # 256 rows x one 256-wide tile per pair; the last N tile leaves rank 1's W half past N
        n_tiles = 8
        m_units = -(-3 * (sms // 2) // n_tiles)
        return m_units * 256 - 200, (n_tiles - 1) * 256 + 96, 320, 0, 0, 256, 256, 1, 2
    # softmax: a cluster of group / 256 CTAs shares one 128-row block and the group's neighbouring 256-wide tiles
    group, valid, N = {"softmax_c1": (128, 100, 512), "softmax_c2": (512, 512, 1024),
                       "softmax_c4": (1024, 1000, 2048)}[kind]
    cs = max(1, group // 256)
    per_row = N // 256 // cs
    m_tiles = -(-3 * (sms // cs) // per_row)
    return m_tiles * 128 - 77, N, 128, group, valid, 128, 256, cs, cs


MULTI_TILE = [(k, e) for k in ("small_n", "single", "pair") for e in range(5)] + \
             [("softmax_c1", 5), ("softmax_c2", 5), ("softmax_c4", 5)]


@pytest.mark.parametrize("kind,epi", MULTI_TILE)
def test_linear_tcgen05_several_tiles_per_cta(ops, kind, epi):
    """Every persistent CTA / cluster works through >= 3 tiles, so the second TMEM accumulator, the accumulator and
    shared-memory ring phases carried from one tile into the next, the parity of the staged bf16 TMA stores and the
    softmax statistics barrier on a cluster's later tiles all run under an fp64 check (reference: DGEMM on the
    device, same bf16 operands)."""
    M, N, K, group, valid, rows, bn, per_unit, cs = _multi_tile_shape(kind)
    assert _tiles_per_unit(M, N, rows, bn, per_unit, cs) >= 3
    g = torch.Generator(device="cuda").manual_seed(M + N + K + epi)
    if epi == 5:
        a = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
        w = (torch.randn(N, K, device="cuda", generator=g) * (4.0 / math.sqrt(K))).to(torch.bfloat16)
        logits = (a.double() @ w.double().T).reshape(M, N // group, group)
        logits[:, :, valid:] = -float("inf")
        want = torch.softmax(logits, dim=-1).reshape(M, N)
        got = ops.linear(a, w, None, 5, None, torch.bfloat16, group=group, group_valid=valid).double()
        assert torch.all(got.reshape(M, N // group, group)[:, :, valid:] == 0)
        torch.testing.assert_close(got, want, atol=2e-3, rtol=1.0e-2)
        return
    a = (torch.randn(M, K, device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g) * 0.1
    res = torch.randn(M, N, device="cuda", generator=g) if epi == 3 else None
    want = _ref_linear(a, w, bias, epi, res)
    for out_dtype in (torch.float32, torch.bfloat16):
        y = ops.linear(a, w, bias, epi, res, out_dtype)
        assert y.dtype == out_dtype and y.shape == want.shape
        tol = 2e-4 if out_dtype == torch.float32 else 1.2e-2
        torch.testing.assert_close(y.double(), want, atol=tol, rtol=tol)


@pytest.mark.parametrize("M,N,K", [(300, 384, 128), (129, 96, 64)])  # CTA pair with a partial tile; small-N
@pytest.mark.parametrize("precision", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("epi", [0, 3, 4])
def test_linear_strided_operands(M, N, K, precision, epi):
    """nrb_linear on column slices of wider buffers: a, w, res and y each have a leading dimension (in elements)
    larger than their width; the columns of y's buffer outside the slice keep their sentinel."""
    from news_recommendation_project_v2_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(M + N + K + epi)
    a = (torch.randn(M, K + 72, device="cuda", generator=g) * 0.5).to(precision)[:, 8:8 + K]
    w = (torch.randn(N, K + 40, device="cuda", generator=g) / math.sqrt(K)).to(precision)[:, 16:16 + K]
    bias = torch.randn(N, device="cuda", generator=g) * 0.1
    res = torch.randn(M, N + 12, device="cuda", generator=g)[:, 4:4 + N] if epi == 3 else None
    want = _ref_linear(a, w, bias, epi, res)
    n_out = want.shape[1]
    for out_dtype in (torch.float32, torch.bfloat16):
        ybuf = torch.full((M, n_out + 24), 12345.0, device="cuda").to(out_dtype)
        before = ybuf.clone()
        y = ybuf[:, 8:8 + n_out]
        _lib.check(_lib.load().nrb_linear(
            _lib.dtype_code(precision), epi, _lib.dtype_code(out_dtype), a.data_ptr(), a.stride(0), w.data_ptr(),
            w.stride(0), bias.data_ptr(), None if res is None else res.data_ptr(), 0 if res is None else res.stride(0),
            y.data_ptr(), y.stride(0), M, N, K, 0, 0, torch.cuda.current_stream().cuda_stream), "nrb_linear")
        if out_dtype == torch.bfloat16:
            tol = 1.2e-2
        else:
            tol = 2e-4 if precision == torch.bfloat16 else 2e-5
        torch.testing.assert_close(y.double(), want, atol=tol, rtol=tol)
        assert torch.equal(ybuf[:, :8], before[:, :8]) and torch.equal(ybuf[:, 8 + n_out:], before[:, 8 + n_out:])


@pytest.mark.parametrize("M,N,K", [(300, 512, 128), (1000, 96, 64)])  # CTA pair, small-N
@pytest.mark.parametrize("epi", [2, 4])
def test_linear_tcgen05_epilogue_full_range(ops, M, N, K, epi):
    """EXP with pre-activations spread over [-60, 60] (relative error, 26 decades), GEGLU with values and gates over
    [-8, 8] (the tails of the erfc polynomial); the spread comes from the bias, the product stays O(0.1)."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K + epi)
    a = (torch.randn(M, K, device="cuda", generator=g) * 0.3).to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
    span = 60.0 if epi == 2 else 8.0
    bias = (torch.rand(N, device="cuda", generator=g) * 2 - 1) * span
    bias[:4] = torch.tensor([-span, span, -span, span])  # both ends in a value and a gate column
    pre = a.double() @ w.double().T + bias.double()
    assert pre.min() < -0.95 * span and pre.max() > 0.95 * span
    want = _ref_linear(a, w, bias, epi, None)
    for out_dtype in (torch.float32, torch.bfloat16):
        y = ops.linear(a, w, bias, epi, None, out_dtype).double()
        if epi == 2:  # relative: one fp32 rounding of the pre-activation at |x| <= 60 costs ~2e-6
            rtol, atol = (2e-5, 0.0) if out_dtype == torch.float32 else (4e-3, 0.0)
        else:  # |y| <= 64; erfc polynomial 1.5e-7 absolute, times |a g|
            rtol, atol = (5e-5, 5e-5) if out_dtype == torch.float32 else (4e-3, 1e-4)
        torch.testing.assert_close(y, want, atol=atol, rtol=rtol)


@pytest.mark.parametrize("M,N,K", [(128, 128, 16), (1, 8, 16), (300, 768, 1024), (257, 4096, 768), (131, 136, 48)])
@pytest.mark.parametrize("epi", [0, 1, 2, 3, 4])
def test_linear_fp32_ffma(ops, M, N, K, epi):
    g = torch.Generator().manual_seed(M + N * 3 + K + epi)
    a = torch.randn(M, K, generator=g) * 0.5
    w = torch.randn(N, K, generator=g) / math.sqrt(K)
    bias = torch.randn(N, generator=g) * 0.1
    res = torch.randn(M, N, generator=g) if epi == 3 else None
    want = _ref_linear(a, w, bias, epi, res)
    y = ops.linear(a.cuda(), w.cuda(), bias.cuda(), epi, None if res is None else res.cuda(), torch.float32)
    torch.testing.assert_close(y.cpu().double(), want, atol=2e-5, rtol=2e-5)  # fp32 FFMA accumulation
    yb = ops.linear(a.cuda(), w.cuda(), bias.cuda(), epi, None if res is None else res.cuda(), torch.bfloat16)
    torch.testing.assert_close(yb.cpu().double(), want, atol=1.2e-2, rtol=1.2e-2)


@pytest.mark.parametrize("precision,tol", [(torch.float32, 2e-5), (torch.bfloat16, 4e-2)])
def test_final_attention_rows_vs_oracle(ops, precision, tol):
    dim, hidden, n = 768, 4096, 700
    sd = syn.make_final_attention_state_dict(dim, hidden, seed=21)
    table = syn.make_table(n, dim, seed=22)
    want_x, want_logit = oracle.final_attention_rows(sd, table, dtype=torch.float64)
    w = {k: (v.to(precision) if k.endswith("weight") else v.float()).cuda().contiguous() for k, v in sd.items()}
    x, e = ops.final_attention_rows(table.to(precision).cuda(), w, torch.float32)
    # fp32: FFMA accumulation noise; bf16: three to five chained bf16 contractions (rel 2^-8 each)
    torch.testing.assert_close(x.cpu().double(), want_x, atol=tol, rtol=tol)
    torch.testing.assert_close(e.cpu().double(), torch.exp(want_logit), atol=tol, rtol=tol)
    xb, eb = ops.final_attention_rows(table.to(precision).cuda(), w, torch.bfloat16)
    torch.testing.assert_close(xb.float().cpu().double(), want_x, atol=max(tol, 1e-2), rtol=max(tol, 1e-2))
    assert eb.dtype == torch.bfloat16


@pytest.mark.parametrize("M,N,K,group,valid", [
    (300, 512, 128, 32, 32), (300, 512, 128, 64, 40), (257, 512, 64, 128, 128), (130, 512, 128, 128, 100),
    (300, 512, 128, 256, 256), (300, 768, 128, 256, 130),          # group == one 256-column tile
    (700, 1024, 256, 512, 512), (129, 4096, 768, 512, 512),        # cluster of 2 (BASELINE L=512)
    (520, 2048, 128, 1024, 1000),                                  # cluster of 4 (BASELINE cfg 5, L=1024)
])
def test_linear_softmax_epilogue_cluster(ops, M, N, K, group, valid):
    """Per-group softmax fused behind the contraction; groups wider than a tile span a CTA cluster (DSMEM)."""
    g = torch.Generator().manual_seed(M + N + K + group + valid)
    a = (torch.randn(M, K, generator=g)).to(torch.bfloat16)
    w = (torch.randn(N, K, generator=g) * (4.0 / math.sqrt(K))).to(torch.bfloat16)  # logits with a real spread
    logits = (a.double() @ w.double().T).reshape(M, N // group, group)
    logits[:, :, valid:] = -float("inf")
    want = torch.softmax(logits, dim=-1).reshape(M, N)
    y = ops.linear(a.cuda(), w.cuda(), None, 5, None, torch.bfloat16, group=group, group_valid=valid)
    got = y.float().cpu().double()
    assert torch.all(got.reshape(M, N // group, group)[:, :, valid:] == 0)
    torch.testing.assert_close(got, want, atol=2e-3, rtol=1.0e-2)  # one bf16 rounding of p in [0,1]
    torch.testing.assert_close(got.reshape(M, N // group, group).sum(-1), torch.ones(M, N // group, dtype=torch.float64),
                               atol=6e-3, rtol=0)
