"""GPU parity tests (B200): every call goes through the C ABI of libcurate_b200.so.

Integer / byte stages are compared bit-exactly with the oracle where the arithmetic is pinned
(colour conversion, frame indices), within the stated fp32-summation budget where it is not
(u8 stage of the antialiased resize: <= 1 LSB on <= 1e-4 of the pixels - the same budget the
oracle itself needs against ATen, tests/test_oracle_cpu.py).  Floating-point stages: tolerance in
each test.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import golden_json, load_golden
from gpu_helpers import ctx, nv12_pool as _nv12_pool, u8_budget as _u8_budget  # noqa: F401
from oracle import color, preprocess, vit

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------ GEMM / LN / attention
@pytest.mark.parametrize(("m", "n", "k"), [(128, 128, 64), (300, 256, 192), (1000, 1024, 1024), (2570, 3072, 1024), (20000, 1024, 4096), (257, 136, 72), (40000, 4096, 1024)])
def test_gemm_plain(ctx, m, n, k):
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    a = (torch.randn(m, k, device="cuda", generator=g) * 0.5).half()
    w = (torch.randn(n, k, device="cuda", generator=g) * 0.5).half()
    bias = torch.randn(n, device="cuda", generator=g)
    got = ctx.gemm(a, w, bias=bias).float()
    want = a.float() @ w.float().T + bias
    err = (got - want).abs().max().item()
    scale = want.abs().max().item()
    assert err <= 2e-3 * scale + 1e-2, (err, scale)  # fp16 output rounding of values ~ sqrt(k)/4


def test_gemm_epilogues(ctx):
    g = torch.Generator(device="cuda").manual_seed(3)
    m, n, k = 3000, 512, 256
    a = (torch.randn(m, k, device="cuda", generator=g) * 0.3).half()
    w = (torch.randn(n, k, device="cuda", generator=g) * 0.2).half()
    bias = torch.randn(n, device="cuda", generator=g)
    z = a.float() @ w.float().T + bias
    from cosmos_curate_b200 import _lib

    got = ctx.gemm(a, w, bias=bias, epilogue=_lib.EPI_QUICK_GELU).float()
    torch.testing.assert_close(got, z * torch.sigmoid(1.702 * z), rtol=2e-3, atol=2e-3)
    got = ctx.gemm(a, w, bias=bias, epilogue=_lib.EPI_GELU_TANH).float()
    torch.testing.assert_close(got, torch.nn.functional.gelu(z, approximate="tanh"), rtol=2e-3, atol=2e-3)
    res = torch.randn(m, n, device="cuda", generator=g)
    want = res + z
    got = ctx.gemm(a, w, bias=bias, residual=res.clone(), out_f32=True)
    torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-3)
    got = ctx.gemm(a, w, out_f32=True)  # no bias, no residual
    torch.testing.assert_close(got, a.float() @ w.float().T, rtol=1e-4, atol=1e-3)


def test_layernorm(ctx):
    g = torch.Generator(device="cuda").manual_seed(4)
    for rows, d in ((1000, 1024), (77, 768), (513, 1152), (9, 256)):
        x = torch.randn(rows, d, device="cuda", generator=g) * 3 + 1
        gamma = torch.randn(d, device="cuda", generator=g)
        beta = torch.randn(d, device="cuda", generator=g)
        got = ctx.layernorm(x, gamma, beta, 1e-5).float()
        want = torch.nn.functional.layer_norm(x, (d,), gamma, beta, 1e-5)
        torch.testing.assert_close(got, want, rtol=2e-3, atol=2e-3)


@pytest.mark.parametrize(("n", "t", "heads", "hd"), [(3, 257, 16, 64), (2, 50, 12, 64), (2, 64, 4, 64), (1, 256, 16, 72), (2, 17, 2, 32),
                                                     (40, 257, 16, 64), (1, 257, 1, 64), (3, 256, 4, 64), (5, 129, 3, 64), (2, 200, 7, 64)])
def test_attention(ctx, n, t, heads, hd):
    g = torch.Generator(device="cuda").manual_seed(t)
    d = heads * hd
    qkv = (torch.randn(n, t, 3 * d, device="cuda", generator=g) * 1.5).half()
    got = ctx.attention(qkv, heads).float()
    q, k, v = qkv.float().view(n, t, 3, heads, hd).permute(2, 0, 3, 1, 4)
    p = torch.softmax(q @ k.transpose(-1, -2) * hd**-0.5, dim=-1)
    want = (p @ v).permute(0, 2, 1, 3).reshape(n, t, d)
    torch.testing.assert_close(got, want, rtol=1e-2, atol=4e-3)  # P and O rounded to fp16




def test_attention_tcgen05_and_mma_kernels_agree(ctx, monkeypatch):
    """head_dim 64 / 129..257 tokens runs on tcgen05 (attention_tc2.cu); CB_ATTN_KERNEL=mma forces the mma.sync kernel."""
    g = torch.Generator(device="cuda").manual_seed(11)
    qkv = (torch.randn(20, 257, 3 * 1024, device="cuda", generator=g) * 2.0).half()
    qkv[:, :, 5] += 6.0  # a dominant query/key channel: sharp softmax rows
    tc = ctx.attention(qkv, 16).float()
    monkeypatch.setenv("CB_ATTN_KERNEL", "mma")
    mma = ctx.attention(qkv, 16).float()
    torch.testing.assert_close(tc, mma, rtol=1e-2, atol=4e-3)
    again = ctx.attention(qkv, 16).float()
    assert torch.equal(mma, again)
    monkeypatch.delenv("CB_ATTN_KERNEL")
    # The tcgen05 kernel issues a tile's four P.V chunk products in the fixed order 0, 2, 1, 3: repeat runs are bitwise equal
    # (also under load: 300 units per CTA-wave with different arrival timing of the two half-row streams).
    for _ in range(3):
        assert torch.equal(tc, ctx.attention(qkv, 16).float())


@pytest.mark.parametrize("kernel", ["1cta", "2cta"])
@pytest.mark.parametrize(("m", "n", "k"), [(300, 256, 192), (257, 136, 72), (1000, 1024, 1024), (5000, 768, 640), (4096, 4304, 1152)])
def test_gemm_both_kernels_with_tails(ctx, monkeypatch, kernel, m, n, k):
    """Force the 1-CTA and the 2-CTA (cta_group::2) kernels through M/N/K tails and the activation epilogue."""
    from cosmos_curate_b200 import _lib

    monkeypatch.setenv("CB_GEMM_KERNEL", kernel)
    g = torch.Generator(device="cuda").manual_seed(m * 7 + n)
    a = (torch.randn(m, k, device="cuda", generator=g) * 0.5).half()
    w = (torch.randn(n, k, device="cuda", generator=g) * 0.5).half()
    bias = torch.randn(n, device="cuda", generator=g)
    z = a.float() @ w.float().T + bias
    got = ctx.gemm(a, w, bias=bias).float()
    assert (got - z).abs().max().item() <= 2e-3 * z.abs().max().item() + 1e-2
    got = ctx.gemm(a, w, bias=bias, epilogue=_lib.EPI_QUICK_GELU).float()
    want = z * torch.sigmoid(1.702 * z)
    assert (got - want).abs().max().item() <= 2e-3 * want.abs().max().item() + 1e-2
    res = torch.randn(m, n, device="cuda", generator=g)
    got = ctx.gemm(a, w, bias=bias, residual=res.clone(), out_f32=True)
    torch.testing.assert_close(got, res + z, rtol=1e-4, atol=2e-3)


@pytest.mark.parametrize(("n", "t", "heads", "hd"), [(2, 729, 16, 72), (1, 600, 4, 64), (1, 1030, 2, 64)])
def test_attention_streamed_keys(ctx, n, t, heads, hd):
    """Sequences whose K/V do not fit shared memory: query tiles split over grid.y, keys streamed in 256-key blocks."""
    g = torch.Generator(device="cuda").manual_seed(t)
    d = heads * hd
    qkv = (torch.randn(n, t, 3 * d, device="cuda", generator=g) * 1.2).half()
    got = ctx.attention(qkv, heads).float()
    q, k, v = qkv.float().view(n, t, 3, heads, hd).permute(2, 0, 3, 1, 4)
    p = torch.softmax(q @ k.transpose(-1, -2) * hd**-0.5, dim=-1)
    want = (p @ v).permute(0, 2, 1, 3).reshape(n, t, d)
    torch.testing.assert_close(got, want, rtol=1e-2, atol=4e-3)
