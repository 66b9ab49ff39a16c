"""GPU parity: the row kernels behind the C entry points nrb_layer_norm, nrb_convert_rows, nrb_split_rows and
nrb_mask_to_csr, each against a plain reference of the same operation (fp64 torch / numpy / torch's own rounding)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from news_recommendation_project_v2_b200 import _lib

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from news_recommendation_project_v2_b200 import ops as _ops
    return _ops


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# (dtype, width, element offset of x): the vector kernels hold NV = width * elemsize / 512 16-byte vectors per lane
# (fp32 NV 1, 2, 3, 4, 6, 8; bf16 NV 1..4); everything else -- fp32 NV 5 and 7, bf16 wider than 1024, widths that are
# no 512-byte multiple, a pointer that is not 16-byte aligned -- runs on the scalar kernel.
LN_CASES = [(torch.float32, d, 0) for d in (128, 256, 384, 512, 768, 1024, 640, 896, 100)] + \
           [(torch.bfloat16, d, 0) for d in (256, 512, 768, 1024, 1280, 2048, 100)] + \
           [(torch.float32, 768, 1), (torch.bfloat16, 1024, 1)]


@pytest.mark.parametrize("dtype,dim,offset", LN_CASES)
@pytest.mark.parametrize("eps", [1e-5, 1e-12])  # LatentAttention / NewAttention
def test_layer_norm_vs_fp64(dtype, dim, offset, eps):
    rows = _sms() * 16 * 8 + 300  # more rows than one grid-stride pass of the 8-warp CTAs
    g = torch.Generator(device="cuda").manual_seed(dim + offset)
    buf = torch.randn(rows, dim + offset, device="cuda", generator=g) * 2 + 0.5
    buf[0] = 3.7  # constant rows: the output is beta
    buf[1] = -1e4 / 3
    buf[2] = 1e4 + 1e-2 * torch.randn(dim + offset, device="cuda", generator=g)  # mean 1e4, spread 1e-2
    buf[3] = -5e3 + 1e-2 * torch.randn(dim + offset, device="cuda", generator=g)
    x = buf.to(dtype)[:, offset:]
    gamma = 1 + 0.1 * torch.randn(dim, device="cuda", generator=g)
    beta = 0.1 * torch.randn(dim, device="cuda", generator=g)
    want = F.layer_norm(x.double(), (dim,), gamma.double(), beta.double(), eps)
    for out_dtype in (torch.float32, torch.bfloat16):
        y = torch.empty(rows, dim, dtype=out_dtype, device="cuda")
        _lib.check(_lib.load().nrb_layer_norm(x.data_ptr(), _lib.dtype_code(dtype), x.stride(0), gamma.data_ptr(),
                                              beta.data_ptr(), eps, y.data_ptr(), _lib.dtype_code(out_dtype),
                                              y.stride(0), rows, dim, torch.cuda.current_stream().cuda_stream),
                   "nrb_layer_norm")
        assert torch.equal(y[:2], beta.to(out_dtype).expand(2, dim))
        if out_dtype == torch.float32:
            torch.testing.assert_close(y.double(), want, atol=1e-5, rtol=1e-5)
        else:  # one bf16 rounding
            torch.testing.assert_close(y.double(), want, atol=1e-3, rtol=4e-3)


def _special_f32():
    """Values where an fp32 -> bf16 rounding goes wrong: ties (even / odd), +-0, +-inf, subnormals, overflow, NaN."""
    bits = np.array([0x3F808000, 0x3F818000, 0xBF808000, 0xBF818000,  # ties: to even (down, up)
                     0x3F807FFF, 0x3F808001,                          # just below / above a tie
                     0x00000000, 0x80000000, 0x7F800000, 0xFF800000,  # +-0, +-inf
                     0x00000001, 0x80000001, 0x00008000, 0x00018000,  # subnormals, subnormal ties
                     0x007FFFFF, 0x00800000, 0x7F7FFFFF, 0xFF7FFFFF,  # largest subnormal, smallest normal, max
                     0x7F7F8000, 0x7F7F7FFF,                          # overflow to inf on the tie, not below
                     0x7FC00000, 0xFFC00001, 0x7F800001], dtype=np.uint32)  # NaNs (quiet, signalling)
    return torch.from_numpy(bits.view(np.float32).copy())


def _assert_bf16_rounding(got, src):
    want = src.to(torch.bfloat16)
    nan = torch.isnan(src)
    assert torch.isnan(got[nan]).all()
    assert torch.equal(got[~nan].view(torch.int16), want[~nan].view(torch.int16))


@pytest.mark.parametrize("dim,offset", [(64, 0), (1000, 0), (100, 0), (64, 1)])  # vector, vector, scalar, scalar
def test_convert_rows_f32_to_bf16_bit_exact(ops, dim, offset):
    rows = 777
    g = torch.Generator(device="cuda").manual_seed(dim)
    buf = torch.randn(rows, dim + offset, device="cuda", generator=g) * \
        torch.exp2(torch.randint(-140, 120, (rows, dim + offset), device="cuda", generator=g).float())
    sp = _special_f32().cuda()
    buf.view(-1)[:sp.numel()] = sp
    buf.view(-1)[-sp.numel():] = sp
    src = buf[:, offset:]
    got = ops.convert_rows(src, torch.bfloat16)
    _assert_bf16_rounding(got, src)


def test_convert_rows_bf16_to_f32_exact_and_strided_destination(ops):
    g = torch.Generator(device="cuda").manual_seed(3)
    src = (torch.randn(513, 136, device="cuda", generator=g) * 100).to(torch.bfloat16)
    src.view(-1)[:7] = torch.tensor([0.0, -0.0, float("inf"), -float("inf"), 1e-40, -3e-39, 2.0 ** 120],
                                    dtype=torch.bfloat16)
    assert torch.equal(ops.convert_rows(src, torch.float32).view(torch.int32), src.float().view(torch.int32))
    # strided destination (ops.pad_rows_for_kernel's layout): the padding columns are never written
    for dst_dtype in (torch.bfloat16, torch.float32):
        for s in (src, src.float()):
            buf = torch.full((513, 256), 7.0, device="cuda", dtype=dst_dtype)
            ops.convert_rows(s, dst_dtype, out=buf[:, :136])
            assert torch.equal(buf[:, :136], s.to(dst_dtype)) and torch.all(buf[:, 136:] == 7.0)


@pytest.mark.parametrize("role", [0, 1])
def test_split_rows_hi_lo_bit_exact(ops, role):
    """hi = bf16(v), lo = bf16(v - hi); role 0 writes [hi | hi | lo], role 1 [hi | lo | hi]."""
    rows, K = 1001, 200
    g = torch.Generator(device="cuda").manual_seed(role)
    src = torch.randn(rows, K, device="cuda", generator=g) * \
        torch.exp2(torch.randint(-60, 60, (rows, K), device="cuda", generator=g).float())
    src.view(-1)[:6] = _special_f32()[:6].cuda()  # ties of the hi rounding
    out = ops.split_rows(src, role)
    hi = src.to(torch.bfloat16)
    lo = (src - hi.float()).to(torch.bfloat16)
    blocks = [hi, hi, lo] if role == 0 else [hi, lo, hi]
    assert out.shape == (rows, 3 * K)
    for b in range(3):
        assert torch.equal(out[:, b * K:(b + 1) * K].view(torch.int16), blocks[b].view(torch.int16)), b


@pytest.mark.parametrize("seq", [1, 31, 33, 100])
def test_mask_to_csr_vs_numpy(ops, seq):
    """More than 1,024 items: the single-CTA scan carries its running total from one block of 1,024 into the next."""
    B = 3001
    rng = np.random.default_rng(seq)
    mask = (rng.random((B, seq)) < rng.random((B, 1))).astype(np.int32)
    mask[::7] = 0  # empty items
    mask[3::11] = 1  # full items
    mask[-1] = 1
    idx, off = ops.mask_to_csr(torch.from_numpy(mask).cuda())
    off = off.cpu().numpy()
    want_off = np.zeros(B + 1, dtype=np.int64)
    np.cumsum(mask.sum(1), out=want_off[1:])
    assert np.array_equal(off, want_off)
    assert np.array_equal(idx[:off[B]].cpu().numpy(), np.flatnonzero(mask.ravel()).astype(np.int32))
