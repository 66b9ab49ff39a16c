"""GPU parity: Stage A (latent-attention pooling) vs golden outputs of the reference / the oracle."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle
from news_recommendation_project_v2_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

# Tolerances on the UNIT-NORM pooled embedding (components are O(1/sqrt(d)) ~ 0.03):
#   fp32 path: FFMA accumulation only                       -> 2e-6 abs
#   bf16 path: bf16 operands through 4 chained contractions -> 2e-3 abs (the reference's own
#              fp32-vs-bf16 drift is 4.3e-4 per component with random-init weights, BASELINE.md)
TOL = {"fp32": 3e-6, "bf16": 2e-3}


def _model(dim, L, seed, precision, **kw):
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    m = LatentAttentionModel(dim=dim, num_latents=L, precision=precision, **kw)
    res = m.load_state_dict(syn.make_latent_state_dict(dim, L, seed=seed, **{k: v for k, v in kw.items()}), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    return m.eval()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["latent_cfg1_d768_L512", "latent_default_d1024_L64", "latent_cfg5_d1024_L1024"])
def test_latent_pool_matches_reference_golden(golden_dir, name, precision):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    dim, L, B, S, seed = (int(g[k]) for k in ("dim", "L", "B", "S", "seed"))
    m = _model(dim, L, seed, precision)
    x, mask = syn.make_token_batch(B, S, dim, seed=seed + 1)
    pooled = m(x.cuda(), mask.cuda())
    assert pooled.shape == (B, dim) and pooled.dtype == torch.float32
    np.testing.assert_allclose(pooled.cpu().numpy(), g["pooled"], atol=TOL[precision], rtol=0)
    np.testing.assert_allclose(pooled.norm(dim=-1).cpu().numpy(), 1.0, atol=1e-5)
    # CPU tensors in -> CPU tensor out (get_model_eval does .to(DEVICE) itself, either works)
    pooled_cpu = m(x, mask)
    assert pooled_cpu.device.type == "cpu" and torch.equal(pooled_cpu, pooled.cpu())
    # mask None -> un-pooled, un-normalised [B,S,d] (latent_attention.py:165)
    un = m(x[:1].cuda(), None)
    assert un.shape == (1, S, dim)
    tol_un = 3e-4 if precision == "fp32" else 6e-2  # O(1..10) magnitudes
    np.testing.assert_allclose(un[0].cpu().numpy(), g["unpooled0"], atol=tol_un, rtol=tol_un)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_latent_mask_semantics_and_chunking(precision):
    from news_recommendation_project_v2_b200 import config
    dim, L = 256, 40  # L not a multiple of 32 -> padded latents must be masked out of the softmax
    m = _model(dim, L, 7, precision, heads=4, dim_head=64)
    sd = m.state_dict()
    x, mask = syn.make_token_batch(37, 24, dim, seed=8, min_len=1)
    mask[5] = 0  # all-masked item -> NaN row (0/0), others unaffected
    mask[7, :] = torch.tensor([1, 0] * 12)  # non-prefix mask pattern
    want = oracle.latent_pool(sd, x, mask, heads=4, dim_head=64, dtype=torch.float64).float()
    old = config.LATENT_MAX_TOKENS
    try:
        outs = []
        for mt in (24, 100, 65536):  # chunk = 1 item, 4 items, everything
            config.LATENT_MAX_TOKENS = mt
            outs.append(m(x.cuda(), mask.cuda()).cpu())
    finally:
        config.LATENT_MAX_TOKENS = old
    for o in outs:
        assert torch.isnan(o[5]).all()
        keep = [i for i in range(37) if i != 5]
        np.testing.assert_allclose(o[keep].numpy(), want[keep].numpy(), atol=TOL[precision] * 2, rtol=0)
    assert torch.equal(outs[0][keep], outs[1][keep]) and torch.equal(outs[1][keep], outs[2][keep])  # chunking is invisible
    # padded tokens never influence the result (SURVEY 3.2): bit-identical output
    x2 = x.clone()
    x2[mask == 0] = 123.0
    assert torch.equal(m(x2.cuda(), mask.cuda()).cpu()[keep], outs[2][keep])
    # bf16 activations are accepted too
    ob = m(x.to(torch.bfloat16).cuda(), mask.cuda()).cpu()
    np.testing.assert_allclose(ob[keep].numpy(), want[keep].numpy(), atol=4e-3, rtol=0)


def test_latent_fold_matches_oracle_projection():
    """A = K_h Wq_h * dh^-0.5 and B = Wout_h V_h^T against fp64."""
    from news_recommendation_project_v2_b200 import ops
    dim, L, heads, dh = 128, 40, 4, 32
    sd = syn.make_latent_state_dict(dim, L, heads=heads, dim_head=dh, seed=3)
    fw = ops.latent_fold(sd, heads, dh, torch.float32, torch.device("cuda"))
    Lp = fw.latents_padded
    assert Lp == 64
    d64 = {k: v.double() for k, v in sd.items()}
    cn = oracle._layer_norm(d64["latents"], d64["cross_attend_blocks.0.norm_context.weight"],
                            d64["cross_attend_blocks.0.norm_context.bias"])
    kv = cn @ d64["cross_attend_blocks.0.fn.to_kv.weight"].T
    inner = heads * dh
    k, v = kv[:, :inner], kv[:, inner:]
    wq, wo = d64["cross_attend_blocks.0.fn.to_q.weight"], d64["cross_attend_blocks.0.fn.to_out.weight"]
    A = torch.zeros(heads * Lp, dim, dtype=torch.float64)
    Bm = torch.zeros(dim, heads * Lp, dtype=torch.float64)
    for h in range(heads):
        sl = slice(h * dh, (h + 1) * dh)
        A[h * Lp:h * Lp + L] = (k[:, sl] @ wq[sl, :]) / dh ** 0.5
        Bm[:, h * Lp:h * Lp + L] = wo[:, sl] @ v[:, sl].T
    torch.testing.assert_close(fw.tensors["a"].cpu().double(), A, atol=1e-5, rtol=1e-5)
    torch.testing.assert_close(fw.tensors["b"].cpu().double(), Bm, atol=1e-5, rtol=1e-5)


def test_refold_after_weight_update():
    m = _model(256, 32, 5, "fp32", heads=2, dim_head=64)
    x, mask = syn.make_token_batch(4, 8, 256, seed=9)
    a = m(x.cuda(), mask.cuda())
    with torch.no_grad():
        m.latents.mul_(1.5)
    b = m(x.cuda(), mask.cuda())
    assert not torch.equal(a, b)
    want = oracle.latent_pool(m.state_dict(), x, mask, heads=2, dim_head=64).float()
    np.testing.assert_allclose(b.cpu().numpy(), want.numpy(), atol=3e-6, rtol=0)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_forward_packed_equals_padded_forward(precision):
    """Varlen entry (packed tokens + CSR offsets) == padded + masked forward, bit for bit; chunked by tokens."""
    from news_recommendation_project_v2_b200 import config
    m = _model(256, 64, 13, precision, heads=4, dim_head=64)
    x, mask = syn.make_token_batch(29, 20, 256, seed=14, min_len=1)
    want = m(x.cuda(), mask.cuda()).cpu()
    lens = mask.sum(1)
    off = torch.zeros(30, dtype=torch.int64)
    off[1:] = torch.cumsum(lens, 0)
    packed = x[mask.bool()]
    old = config.LATENT_MAX_TOKENS
    try:
        for mt in (20, 77, 65536):
            config.LATENT_MAX_TOKENS = mt
            got = m.forward_packed(packed.cuda(), off).cpu()
            assert torch.equal(got, want)
    finally:
        config.LATENT_MAX_TOKENS = old
    assert m.forward_packed(packed, off).device.type == "cpu"


def test_apply_token_attn_from_token_store(tmp_path):
    """Token store -> forward_packed == the reference flow (pad to batch max + mask + forward)."""
    from news_recommendation_project_v2_b200.token_store import apply_token_attn, write_token_store
    m = _model(256, 64, 21, "fp32", heads=4, dim_head=64)
    g = torch.Generator().manual_seed(3)
    items = [torch.randn(int(n), 256, generator=g).half() for n in torch.randint(1, 30, (37,), generator=g)]
    db = str(tmp_path / "tok.sqlite")
    write_token_store(db, items)
    got = apply_token_attn(m, db, len(items), chunk_items=10)
    S = max(t.shape[0] for t in items)
    x = torch.zeros(len(items), S, 256)
    mask = torch.zeros(len(items), S, dtype=torch.int32)
    for i, t in enumerate(items):
        x[i, :t.shape[0]] = t.float()
        mask[i, :t.shape[0]] = 1
    want = oracle.latent_pool(m.state_dict(), x, mask, heads=4, dim_head=64).float()
    # bf16 token storage in read_token_store (default) vs fp16 source: compare at bf16 input precision
    np.testing.assert_allclose(got.numpy(), want.numpy(), atol=2e-3, rtol=0)


def test_packed_token_file_pipeline_equals_padded_forward(tmp_path):
    """Packed token FILE -> pinned double-buffered chunks -> forward_packed == padded + masked forward on the same
    (bf16) tokens, bit for bit, whatever the chunk size; empty items give NaN rows."""
    from news_recommendation_project_v2_b200.token_store import apply_token_attn_packed, write_packed_tokens
    m = _model(256, 64, 21, "bf16", heads=4, dim_head=64)
    g = torch.Generator().manual_seed(5)
    items = [torch.randn(int(n), 256, generator=g).to(torch.bfloat16) for n in torch.randint(1, 40, (83,), generator=g)]
    items[17] = items[17][:0]  # an empty item
    # /dev/shm when there is one: shared-memory pages are what cudaHostRegister accepts (the zero-copy branch below)
    shm = os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK)
    path = "/dev/shm/nrb200_test_%d.nrbtok" % os.getpid() if shm else str(tmp_path / "tok.nrbtok")
    try:
        _packed_file_checks(m, items, path)
    finally:
        if shm and os.path.exists(path):
            os.remove(path)


def _packed_file_checks(m, items, path):
    from news_recommendation_project_v2_b200.token_store import apply_token_attn_packed, write_packed_tokens
    write_packed_tokens(path, items, 256)
    S = max(t.shape[0] for t in items)
    x = torch.zeros(len(items), S, 256, dtype=torch.bfloat16)
    mask = torch.zeros(len(items), S, dtype=torch.int32)
    for i, t in enumerate(items):
        x[i, :t.shape[0]] = t
        mask[i, :t.shape[0]] = 1
    want = m(x.cuda(), mask.cuda()).cpu()
    keep = [i for i in range(len(items)) if i != 17]
    for chunk in (40, 333, 1 << 20):
        got = apply_token_attn_packed(m, path, chunk_tokens=chunk, copy_threads=3)
        assert got.is_pinned() and got.shape == (83, 256)
        assert torch.isnan(got[17]).all() and torch.equal(got[keep], want[keep])
    # zero-copy variant: the mapped token section page-locked for the GPU (skipped if the driver refuses)
    from news_recommendation_project_v2_b200.token_store import PackedTokenFile
    tf = PackedTokenFile(path)
    if tf.register():
        for chunk in (40, 333, 1 << 20):
            got = apply_token_attn_packed(m, tf, chunk_tokens=chunk)
            assert torch.isnan(got[17]).all() and torch.equal(got[keep], want[keep])
        tf.unregister()
    else:
        print("cudaHostRegister refused the mapping:", tf.register_error)


def test_packed_all_empty_items_give_nan():
    """A chunk whose items are all empty returns NaN rows like the reference's 0/0 masked mean, never
    uninitialised memory (ADVICE r1)."""
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    m = LatentAttentionModel(dim=256, num_latents=64, heads=4, dim_head=64, precision="bf16").eval()
    m.load_state_dict(syn.make_latent_state_dict(256, 64, heads=4, dim_head=64, seed=1))
    out = m.forward_packed(torch.zeros(0, 256, device="cuda"), torch.zeros(4, dtype=torch.int64))
    assert out.shape == (3, 256) and torch.isnan(out).all()
    # mixed: empty items between real ones
    g = torch.Generator().manual_seed(0)
    tok = torch.randn(10, 256, generator=g)
    off = torch.tensor([0, 0, 4, 4, 10, 10])
    out = m.forward_packed(tok.cuda(), off).cpu()
    assert torch.isnan(out[[0, 2, 4]]).all() and torch.isfinite(out[[1, 3]]).all()
    want = m.forward_packed(tok.cuda(), torch.tensor([0, 4, 10])).cpu()
    assert torch.equal(out[[1, 3]], want)


def _softmax_gemm_tiles_per_cluster(n_tokens, heads, latents_padded):
    """Tiles per persistent cluster of the fused softmax GEMM over n_tokens rows, the way launch_gemm sizes its grid
    (clusters of Lp / 256 CTAs share a 128-row block; at most SMs / cluster co-resident clusters)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cs = max(1, latents_padded // 256)
    units = -(-n_tokens // 128) * (heads * latents_padded // 256 // cs)
    return units / (sms // cs)


def _token_batch_with_at_least(n_valid, S, dim, seed):
    """Padded token batch [B, S, dim] (prefix masks, 1..S tokens per item) holding at least n_valid tokens."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(1, S + 1, (2 * n_valid // S + 2 * S,), generator=g)
    B = int(torch.searchsorted(torch.cumsum(lens, 0), n_valid).item()) + 1
    lens = lens[:B]
    mask = (torch.arange(S)[None, :] < lens[:, None]).to(torch.int32)
    return torch.randn(B, S, dim, generator=g), mask


def test_latent_stage_a_several_tiles_per_cta():
    """Stage A at scale (bf16, fused softmax GEMM with one 256-column tile per row block): enough valid tokens that
    every CTA works through >= 3 tiles with the device-side row count and row map of the masked path, and more than
    1,024 items in one chunk (the carry of the item-offset scan).  Padded + masked and packed forms against the fp64
    oracle on the device, and bit-equal to each other."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    m = _model(256, 64, 31, "bf16", heads=4, dim_head=64)
    x, mask = _token_batch_with_at_least(3 * sms * 128 + 200, 20, 256, seed=32)
    n_tok = int(mask.sum())
    assert _softmax_gemm_tiles_per_cluster(n_tok, 4, 64) >= 3 and mask.shape[0] > 1024
    from news_recommendation_project_v2_b200 import config
    assert x.shape[0] * x.shape[1] <= config.LATENT_MAX_TOKENS  # one chunk
    sd = {k: v.cuda() for k, v in m.state_dict().items()}
    want = oracle.latent_pool(sd, x.cuda(), mask.cuda(), heads=4, dim_head=64, dtype=torch.float64)
    got = m(x.cuda(), mask.cuda())
    torch.testing.assert_close(got.double(), want, atol=TOL["bf16"], rtol=0)
    off = torch.zeros(mask.shape[0] + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(mask.sum(1), 0)
    packed = m.forward_packed(x[mask.bool()].cuda(), off)
    assert torch.equal(packed, got)


def test_latent_cluster_of_4_several_tiles_per_cluster():
    """d=1024, L=1024 (8 heads x 512): the softmax over 1,024 latents spans a cluster of 4 CTAs; enough tokens that
    each co-resident cluster works through >= 3 row blocks (the statistics barrier on a cluster's later tiles)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    m = _model(1024, 1024, 41, "bf16")
    need = -(-3 * (sms // 4) // 8) * 128  # 8 units per 128-row block
    x, mask = _token_batch_with_at_least(need + 200, 24, 1024, seed=42)
    assert _softmax_gemm_tiles_per_cluster(int(mask.sum()), 8, 1024) >= 3
    sd = {k: v.cuda() for k, v in m.state_dict().items()}
    want = oracle.latent_pool(sd, x.cuda(), mask.cuda(), heads=8, dim_head=512, dtype=torch.float64)
    got = m(x.cuda(), mask.cuda())
    torch.testing.assert_close(got.double(), want, atol=TOL["bf16"], rtol=0)
