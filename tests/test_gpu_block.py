"""GPU parity of the composed hot path: one Wan DiT block (turbodiffusion_b200/block.py) against the CPU oracle's
restatement of WanAttentionBlock.forward after model surgery (oracle.wan_block_forward)."""
import pytest
import torch

from oracle import td_oracle as O

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dim,heads,ffn,thw,lc,topk", [(256, 2, 512, (3, 10, 20), 77, 0.3), (384, 3, 640, (2, 9, 25), 64, 0.5)])
def test_block_matches_oracle(cuda, dim, heads, ffn, thw, lc, topk):
    from turbodiffusion_b200.block import WanBlockB200, random_block_state
    torch.manual_seed(0)
    l = thw[0] * thw[1] * thw[2]
    sd = random_block_state(dim, ffn, heads, seed=3, device=cuda)
    blk = WanBlockB200(sd, dim, heads, topk=topk)
    x = torch.randn(l, dim).bfloat16()
    e0 = torch.randn(6, dim) * 0.1
    ctx = torch.randn(lc, dim).bfloat16()
    ang = O.wan_rope_angles(*thw, dim // heads)
    out = blk(x.to(cuda), e0.to(cuda), ang.to(cuda), ctx.to(cuda)).cpu()
    ref = O.wan_block_forward({k: v.cpu() for k, v in sd.items()}, x, e0, ang, ctx, dim, heads, topk=topk, sla_mode="exact")
    st = O.stats(out, ref)
    assert st["cos"] > 0.9995 and st["rel_l2"] < 2.5e-2, st
    assert out.dtype == x.dtype and out.shape == x.shape


def test_fused_qkv_block_equals_the_unfused_one(cuda, monkeypatch):
    """f2: the q/k/v projections as one split-output GEMM (block.FUSE_QKV) change nothing in the block's output (the
    projections themselves are compared bit for bit in test_split_output_gemm_equals_the_separate_gemms): the two blocks'
    outputs are bit-identical."""
    from turbodiffusion_b200 import block as B
    dim, heads, ffn, thw = 512, 4, 1024, (3, 10, 23)
    l = thw[0] * thw[1] * thw[2]
    sd = B.random_block_state(dim, ffn, heads, seed=9, device=cuda)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(l, dim, generator=g).bfloat16().to(cuda)
    e0 = (torch.randn(6, dim, generator=g) * 0.1).to(cuda)
    ctx = torch.randn(40, dim, generator=g).bfloat16().to(cuda)
    ang = O.wan_rope_angles(*thw, dim // heads).to(cuda)
    outs = {}
    for mode in ("0", "1"):
        monkeypatch.setattr(B, "FUSE_QKV", mode)
        outs[mode] = B.WanBlockB200(sd, dim, heads, topk=0.3)(x, e0, ang, ctx)
    assert torch.equal(outs["0"], outs["1"])


def test_block_keeps_reference_state_dict_keys(cuda):
    from turbodiffusion_b200.block import LINEARS, random_block_state
    sd = random_block_state(256, 512, 2, seed=0, device=cuda)
    for name in LINEARS:
        assert sd[name + ".int8_weight"].dtype == torch.int8 and sd[name + ".scale"].dtype == torch.float32
    assert sd["self_attn.attn_op.local_attn.proj_l.weight"].shape == (128, 128)


def test_missing_library_fails_loudly(monkeypatch, cuda):
    from turbodiffusion_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libtdb200.so")
    with pytest.raises(_lib.Tdb200Error):
        _lib.lib()
