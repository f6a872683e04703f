"""Flash self-attention (ops.flash_attn64) beyond the operator battery of tests/ops_cases.py: shapes that reach the
partial key block, the partial or empty second query tile of a CTA and the batched split-KV grid; logits that make
the lazy O rescale run many times; run-to-run bit reproducibility of the split-KV path."""
import pytest

from tests.ops_cases import case_attn

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("NB,T,C", [(1, 63, 64), (3, 200, 128), (8, 9216, 320)],
                         ids=["t63_less_than_one_block", "nb3_t200_ragged", "nb8_t9216_batched"])
def test_attention_shapes(NB, T, C):
    import torch

    res = case_attn(NB=NB, T=T, C=C)
    torch.cuda.synchronize()
    assert res["ok"], {k: v for k, v in res.items() if k != "ms"}


@pytest.mark.parametrize("NB,T,C", [(1, 2304, 128), (2, 9216, 64), (1, 200, 64)])
def test_attention_growing_logits_rescale(NB, T, C):
    """Row r's logits move along the key sequence by up to s_r * 64 log2 units (s_r in [-1, 1]): the running max of
    the rows with s_r > 0 grows in almost every key block, so O is rescaled many times, next to rows of the same warp
    that never rescale. Random qkv hardly ever crosses the threshold of 8 log2 units after the first block."""
    import math

    import torch
    import torch.nn.functional as F

    from marigold_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(11)
    h = C // 64
    qkv = torch.randn(NB * T, 3 * C, device="cuda", generator=g) * 0.5
    v = qkv.view(NB, T, 3, h, 64)
    span = 64.0 / math.log2(math.e) * 8.0                                   # q . k / 8 = 64 log2 units at s = 1
    s = torch.rand(NB, T, h, device="cuda", generator=g) * 2 - 1
    v[:, :, 0, :, 0] = 16.0 * s
    v[:, :, 1, :, 0] = (span / 16.0) * torch.linspace(0, 1, T, device="cuda")[None, :, None]
    qkv = qkv.to(torch.bfloat16)
    q, k, vv = [t.float().reshape(NB, T, h, 64).permute(0, 2, 1, 3) for t in qkv.split(C, dim=1)]
    ref = F.scaled_dot_product_attention(q, k, vv).permute(0, 2, 1, 3).reshape(NB * T, C)
    out = ops.flash_attn64(qkv, NB, T, C, 0.125).float()
    torch.cuda.synchronize()
    assert not torch.isnan(out).any()
    rel = ((out - ref).abs().max() / ref.abs().max()).item()
    assert rel < 2e-2, rel


def test_attention_split_kv_is_bit_reproducible():
    import torch

    from marigold_b200 import ops

    T, C = 9216, 320   # 180 tile pairs on 148 SMs: the KV range is split and merged by attn_combine_kernel
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = torch.randn(T, 3 * C, device="cuda", generator=g).to(torch.bfloat16)
    a = ops.flash_attn64(qkv, 1, T, C, 0.125).clone()
    b = ops.flash_attn64(qkv, 1, T, C, 0.125)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
