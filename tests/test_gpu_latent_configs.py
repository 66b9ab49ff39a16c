"""GPU parity: stage A (latent-attention pooling) at every softmax layout against fp64.

The bf16 forward runs the per-head softmax either fused into the logits GEMM (a row of Lp columns spread over a
cluster of Lp / 256 CTAs, statistics per 32-column chunk) or unfused (fp32 logits, then `softmax_groups`); the fp32
forward always runs the unfused FFMA path.  Each case below names the layout it runs and asserts it, then checks the
pooled output, one un-pooled item, the packed entry and an all-masked item against the fp64 oracle on the same weights.
The shift tests move every logit far below zero, where a softmax chunk holding only padded columns used to turn into
NaN (softmax is shift invariant, so such logits are legal input).
"""
import math

import pytest
import torch

from oracle import oracle
from news_recommendation_project_v2_b200 import config, synthetic as syn
from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel

pytestmark = pytest.mark.gpu

# Tolerances on the unit-norm pooled embedding, as in test_gpu_latent.py (fp32: FFMA accumulation; bf16: bf16 operands
# through four chained contractions).  Largest pooled error measured on a B200 (1,000 W) over the d = 256 cases of this
# file: fp32 7.9e-7 (the far-below-zero logits, 3.8x headroom; 5.4e-8 elsewhere), bf16 1.5e-4 (13x headroom).
TOL = {"fp32": 3e-6, "bf16": 2e-3}
TOL_UNPOOLED = {"fp32": 3e-4, "bf16": 6e-2}  # per-token block output, O(1..10) magnitudes (atol and rtol)


def _latents_padded(L):
    return max(32, 1 << (L - 1).bit_length())


def _bf16_softmax_layout(heads, Lp):
    """The softmax the bf16 forward runs, decided the way `fused_softmax` in csrc/latent.cu decides it: fused when the
    logits tile into whole 256-column MMA tiles and a row fits one cluster (Lp <= 1024), with Lp / 256 CTAs per
    cluster; otherwise unfused."""
    if heads * Lp % 256 == 0 and Lp <= 1024:
        return "fused", max(1, Lp // 256)
    return "unfused", 0


# (dim, L, heads, dim_head) -> (Lp, heads * Lp, bf16 softmax layout, cluster size)
CASES = {
    # padding inside the only 32-column chunk of each head's group
    "narrow_group": ((256, 20, 8, 32), (32, 256, "fused", 1)),
    # columns 96..127 of each group are all padding: a chunk with no valid column
    "padded_chunk": ((256, 72, 2, 64), (128, 256, "fused", 1)),
    # L not a multiple of 4: the fold rounds its latent rows up to 52
    "l50": ((256, 50, 4, 32), (64, 256, "fused", 1)),
    # the second CTA of each 2-CTA cluster holds 4 valid columns and 7 empty chunks
    "cluster2_4_valid": ((256, 260, 2, 64), (512, 1024, "fused", 2)),
    # cluster of 2 and L % 4 == 1
    "cluster2_409": ((256, 409, 2, 64), (512, 1024, "fused", 2)),
    # the fourth CTA of the 4-CTA cluster holds only padding
    "cluster4_empty_cta": ((256, 600, 1, 64), (1024, 1024, "fused", 4)),
    # the head layout of the reference's 4096-d branch (2 heads x 32, 32 latents): heads * Lp = 64
    "unfused_2x32": ((256, 32, 2, 32), (32, 64, "unfused", 0)),
    # one head, heads * Lp = 128
    "unfused_one_head": ((256, 100, 1, 64), (128, 128, "unfused", 0)),
    # Lp > 1024: a row does not fit one cluster
    "unfused_lp2048": ((256, 1500, 2, 64), (2048, 4096, "unfused", 0)),
}


def _model(dim, L, heads, dh, precision, seed, sd=None):
    m = LatentAttentionModel(dim=dim, num_latents=L, heads=heads, dim_head=dh, precision=precision)
    if sd is None:
        sd = syn.make_latent_state_dict(dim, L, heads=heads, dim_head=dh, seed=seed)
    res = m.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    return m.eval()


def _assert_layout(m, precision, Lp, hl, layout, cluster):
    fw = m.folded()
    assert fw.latents_padded == Lp and fw.heads * fw.latents_padded == hl
    assert fw.latents_padded == _latents_padded(fw.num_latents)
    if precision == "bf16":
        assert _bf16_softmax_layout(fw.heads, fw.latents_padded) == (layout, cluster)


def _check_against_fp64(m, heads, dh, precision, B, S, seed, tol, tag):
    """Pooled output (with one all-masked item) and one un-pooled item against fp64; the packed entry bit-equal to the
    padded one; the all-masked item changes no other row.  Returns the largest pooled error."""
    dim = m.latents.shape[1]
    x, mask_full = syn.make_token_batch(B, S, dim, seed=seed, min_len=1)
    e = B // 2
    mask = mask_full.clone()
    mask[e] = 0
    keep = [i for i in range(B) if i != e]
    sd = {k: v.cuda() for k, v in m.state_dict().items()}
    xd, md = x.cuda(), mask.cuda()
    want = oracle.latent_pool(sd, xd, md, heads=heads, dim_head=dh, dtype=torch.float64)
    got = m(xd, md)
    assert torch.isnan(got[e]).all() and torch.isfinite(got[keep]).all()
    err = (got[keep].double() - want[keep]).abs().max().item()
    # the item's tokens leave the packed rows; every other item's rows and their arithmetic stay the same
    assert torch.equal(m(xd, mask_full.cuda())[keep], got[keep])
    # varlen entry: the same packed rows, bit for bit
    off = torch.zeros(B + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(mask.sum(1), 0)
    packed = m.forward_packed(x[mask.bool()].cuda(), off)
    assert torch.isnan(packed[e]).all() and torch.equal(packed[keep], got[keep])
    # un-pooled (mask None): every position of one item, padded ones included
    un = m(xd[:1], None)
    want_un = oracle.latent_block(sd, xd[:1], heads=heads, dim_head=dh, dtype=torch.float64)
    err_un = (un.double() - want_un).abs().max().item()
    print(f"{tag} {precision}: pooled max err {err:.2e} (tol {tol:.0e}), un-pooled max err {err_un:.2e}")
    torch.testing.assert_close(got[keep].double(), want[keep], atol=tol, rtol=0)
    tu = TOL_UNPOOLED[precision]
    torch.testing.assert_close(un.double(), want_un, atol=tu, rtol=tu)
    return err


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", list(CASES))
def test_latent_layout_vs_fp64(case, precision):
    (dim, L, heads, dh), (Lp, hl, layout, cluster) = CASES[case]
    m = _model(dim, L, heads, dh, precision, seed=L + heads)
    _assert_layout(m, precision, Lp, hl, layout, cluster)
    _check_against_fp64(m, heads, dh, precision, B=24, S=16, seed=L + 1, tol=TOL[precision], tag=case)


@pytest.fixture(scope="module")
def model_4096():
    """The model the reference builds when EMBEDDING_DIM is 4096: dim from the config, 32 latents, 2 heads x 32
    (latent_attention.py:91-104), with synthetic weights."""
    old = config.EMBEDDING_DIM, config.REDUCED_DIM
    config.EMBEDDING_DIM = config.REDUCED_DIM = 4096
    try:
        m = LatentAttentionModel()
    finally:
        config.EMBEDDING_DIM, config.REDUCED_DIM = old
    attn = m.cross_attend_blocks[0].fn
    assert (m.latents.shape, attn.heads, attn.dim_head) == ((32, 4096), 2, 32)
    m.load_state_dict(syn.make_latent_state_dict(4096, 32, heads=2, dim_head=32, seed=4096), strict=True)
    return m.eval()


# d = 4096: unit-norm components are half the size they are at d = 1024, and the bf16 error shrinks with them.  Measured
# on a B200 (1,000 W): fp32 3.6e-8, bf16 4.0e-5, so the bf16 bound is 2e-4 (5x headroom) instead of 2e-3.
@pytest.mark.parametrize("precision,tol", [("fp32", 3e-6), ("bf16", 2e-4)])
def test_latent_reference_4096_branch_vs_fp64(model_4096, precision, tol):
    """dim 4096 (the widest row `pool_items_kernel<4>` holds), a 32,768-wide GEGLU and the unfused softmax."""
    m = model_4096
    m.precision = precision
    _assert_layout(m, precision, 32, 64, "unfused", 0)
    _check_against_fp64(m, 2, 32, precision, B=16, S=24, seed=4097, tol=tol, tag="ref_4096")


@pytest.mark.parametrize("offset", [-120.0, 0.0, 120.0])
@pytest.mark.parametrize("group,valid", [(64, 20), (128, 72), (512, 260), (1024, 600)])
def test_softmax_epilogue_empty_chunks_under_shift(group, valid, offset):
    """Fused softmax epilogue with groups that hold at least one 32-column chunk of padding only, all logits moved by
    `offset`.  At -120 every row's largest valid logit is below -88.7, where 2^(-max * log2 e) overflows fp32."""
    from news_recommendation_project_v2_b200 import ops
    assert group - valid >= 32
    M, K = 300, 128
    N = 2 * max(group, 256)
    g = torch.Generator(device="cuda").manual_seed(group + valid)
    a = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda", generator=g) * (4.0 / math.sqrt(K))).to(torch.bfloat16)
    a[:, 0] = 1.0
    w[:, 0] = offset  # exact in bf16: the same shift on every logit
    logits = (a.double() @ w.double().T).reshape(M, N // group, group)
    if offset < 0:
        assert logits[:, :, :valid].max() < -88.7
    logits[:, :, valid:] = -float("inf")
    want = torch.softmax(logits, dim=-1).reshape(M, N)
    got = ops.linear(a, w, None, 5, None, torch.bfloat16, group=group, group_valid=valid).double()
    assert torch.all(got.reshape(M, N // group, group)[:, :, valid:] == 0)
    torch.testing.assert_close(got, want, atol=2e-3, rtol=1.0e-2)  # one bf16 rounding of p in [0, 1]
    torch.testing.assert_close(got.reshape(M, N // group, group).sum(-1),
                               torch.ones(M, N // group, dtype=torch.float64, device="cuda"), atol=6e-3, rtol=0)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("L,heads,dh", [(72, 2, 64), (600, 1, 64)])
def test_latent_logits_far_below_zero(L, heads, dh, precision):
    """Every logit of every head is -100: LN1 with weight 0 and bias -100 u gives every token the same normalised
    input, LN_ctx with weight 0 and bias v gives every latent the same key, and each head's block of to_q is scaled so
    that its (u, v) logit is -100.  The softmax is uniform; on the fused path the padded chunks of these layouts
    (columns 96..127 of 128; the fourth CTA of a 4-CTA cluster) must contribute exactly 0."""
    dim = 256
    sd = syn.make_latent_state_dict(dim, L, heads=heads, dim_head=dh, seed=L + 5)
    g = torch.Generator().manual_seed(L + 6)
    u, v = torch.randn(dim, generator=g), torch.randn(dim, generator=g)
    p0 = "cross_attend_blocks.0."
    inner = heads * dh
    wq, wk = sd[p0 + "fn.to_q.weight"], sd[p0 + "fn.to_kv.weight"][:inner]
    for h in range(heads):
        sl = slice(h * dh, (h + 1) * dh)
        c = float((u.double() @ wq[sl].double().T) @ (v.double() @ wk[sl].double().T)) / math.sqrt(dh)
        wq[sl] /= c
    sd[p0 + "norm.weight"] = torch.zeros(dim)
    sd[p0 + "norm.bias"] = -100.0 * u
    sd[p0 + "norm_context.weight"] = torch.zeros(dim)
    sd[p0 + "norm_context.bias"] = v
    q = (-100.0 * u.double()) @ wq.double().T
    k = v.double() @ wk.double().T
    logits = (q.view(heads, dh) * k.view(heads, dh)).sum(-1) / math.sqrt(dh)
    torch.testing.assert_close(logits, torch.full((heads,), -100.0, dtype=torch.float64), atol=1e-3, rtol=0)
    m = _model(dim, L, heads, dh, precision, seed=0, sd=sd)
    if precision == "bf16":
        assert _bf16_softmax_layout(heads, _latents_padded(L))[0] == "fused"
    _check_against_fp64(m, heads, dh, precision, B=24, S=16, seed=L + 7, tol=TOL[precision], tag=f"shift_L{L}")


def test_bf16_rejects_heads_times_padded_latents_not_multiple_of_64():
    """One head of 32 padded latents: the bf16 value GEMM would contract over K = 32, which the tensor-core GEMM does
    not take.  The fold refuses the layout by name; the same weights run in fp32 and match fp64."""
    from news_recommendation_project_v2_b200 import _lib, ops
    dim, L, heads, dh = 256, 32, 1, 64
    sd = syn.make_latent_state_dict(dim, L, heads=heads, dim_head=dh, seed=33)
    with pytest.raises(_lib.NrbError, match=r"heads \* latents_padded .*\(got 1 x 32\)"):
        ops.latent_fold(sd, heads, dh, torch.bfloat16, torch.device("cuda"))
    with pytest.raises(_lib.NrbError, match=r"heads \* latents_padded"):
        _model(dim, L, heads, dh, "bf16", seed=0, sd=sd)(torch.zeros(1, 4, dim, device="cuda"),
                                                        torch.ones(1, 4, dtype=torch.int32, device="cuda"))
    m = _model(dim, L, heads, dh, "fp32", seed=0, sd=sd)
    _check_against_fp64(m, heads, dh, "fp32", B=24, S=16, seed=34, tol=TOL["fp32"], tag="one_head_32")
