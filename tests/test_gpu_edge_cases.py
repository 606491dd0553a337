"""Edge cases of the hot path through the public operator API: empty inputs, key sequences shorter than one reduction chunk,
checkpoint-dtype (bf16) side inputs.  The reference's own tests exercise none of these shapes; its operators either return
empty tensors (torch semantics) or are only defined for l >= 1."""
import pytest
import torch

from oracle import td_oracle as O

pytestmark = pytest.mark.gpu


def test_empty_inputs_return_empty_outputs(cuda):
    import turbodiffusion_b200.ops as ops
    from turbodiffusion_b200.turbo_diffusion_ops import gemm_cuda_swizzle_bias, quant_cuda
    x0 = torch.empty(0, 256, dtype=torch.bfloat16, device=cuda)
    q, s = quant_cuda(x0)
    assert q.shape == (0, 256) and s.shape == (0, 2)
    w_q, w_s = ops.int8_quant((torch.randn(128, 256) * 0.1).bfloat16().to(cuda))
    y = torch.empty(0, 128, dtype=torch.bfloat16, device=cuda)
    gemm_cuda_swizzle_bias(q, s, w_q, w_s, y, None)                     # m = 0: nothing to launch, no error
    assert ops.fast_rmsnorm(x0, torch.ones(256, device=cuda), 1e-6).shape == (0, 256)
    assert ops.fast_layernorm(x0, None, None, 1e-6).shape == (0, 256)
    lin = ops.Int8Linear.from_linear(torch.nn.Linear(256, 128).to(cuda).bfloat16(), quantize=True)
    assert lin(x0).shape == (0, 128)
    torch.cuda.synchronize()


@pytest.mark.parametrize("lk", [1, 2, 3, 5, 127, 129])
def test_key_sequences_shorter_than_a_reduction_chunk(cuda, lk):
    """ADVICE r1: the key-mean partial sums used to be staged in the INT8 output buffer, too small for lk < 4.  One 128-row
    chunk now reduces straight into the kmean output; codes, scales and pooled means stay exact vs the Sage emulation."""
    from turbodiffusion_b200.SLA.utils import quant_qk
    g = torch.Generator().manual_seed(lk)
    q = torch.randn(1, 200, 2, 128, generator=g).bfloat16()
    k = (torch.randn(1, lk, 2, 128, generator=g) + 1.5).bfloat16()
    guard = torch.full((1, 2, lk + 64, 128), 77, dtype=torch.int8, device=cuda)       # rows past lk must stay untouched
    prep = quant_qk(q.to(cuda), k.to(cuda))
    torch.cuda.synchronize()
    kh = k.transpose(1, 2).contiguous()
    torch.testing.assert_close(prep.kmean.cpu(), kh.float().mean(-2), rtol=1e-5, atol=1e-5)
    arg_k = kh - prep.kmean.cpu().to(k.dtype)[:, :, None, :]
    k_i8, k_s = O.sage_quant_blocks(arg_k, 64)
    assert torch.equal(prep.k_scale.cpu(), k_s) and torch.equal(prep.k_i8.cpu(), k_i8)
    assert prep.k_i8.shape == (1, 2, lk, 128) and (guard == 77).all()


def test_sla_forward_on_a_sequence_of_one_key_block(cuda):
    """L < 64: a single ragged key block, topk clamps to 1 (the reference's int(topk*nblk) would be 0 and its softmax empty)."""
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    g = torch.Generator().manual_seed(3)
    q, k, v = (torch.randn(1, 37, 2, 128, generator=g).bfloat16() for _ in range(3))
    m = SageSparseLinearAttention(128, 0.1).to(cuda)
    with torch.no_grad():
        m.proj_l.weight.normal_(0, 0.05)
        m.proj_l.bias.normal_(0, 0.05)
    out = m(q.to(cuda), k.to(cuda), v.to(cuda)).cpu()
    ref = O.sla_forward(q, k, v, m.proj_l.weight.cpu(), m.proj_l.bias.cpu(), 1.0, mode="sage")     # every (= the only) block
    st = O.stats(out, ref)
    assert st["cos"] > 0.999 and st["rel_l2"] < 2e-2, st


def test_checkpoint_dtype_side_inputs_are_converted_not_reinterpreted(cuda):
    """ADVICE r1: load_state_dict(assign=True) keeps norm weights / modulation in the checkpoint's bf16.  The fused entry points
    read fp32 pointers, so the shims must convert: a bf16 weight gives exactly the result of its fp32 copy."""
    import turbodiffusion_b200.ops as ops
    from turbodiffusion_b200.block import WanBlockB200, random_block_state
    dim, heads, ffn, thw = 256, 2, 512, (2, 6, 10)
    l = thw[0] * thw[1] * thw[2]
    g = torch.Generator().manual_seed(5)
    x = torch.randn(l, dim, generator=g).bfloat16().to(cuda)
    w16 = (torch.rand(dim, generator=g) + 0.5).bfloat16().to(cuda)
    ang = O.wan_rope_angles(*thw, dim // heads).to(cuda)
    assert torch.equal(ops.rmsnorm_rope(x, w16, ang, 1e-6, heads), ops.rmsnorm_rope(x, w16.float(), ang, 1e-6, heads))
    assert torch.equal(ops.fast_rmsnorm(x, w16, 1e-6), ops.fast_rmsnorm(x, w16.float(), 1e-6))
    sc16, sh16 = (torch.randn(dim, generator=g) * 0.1).bfloat16().to(cuda), (torch.randn(dim, generator=g) * 0.1).bfloat16().to(cuda)
    a, b = ops.layernorm_modulate_quant(x, sc16, sh16, 1e-6), ops.layernorm_modulate_quant(x, sc16.float(), sh16.float(), 1e-6)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(ops.gate_residual(x, x, sc16), ops.gate_residual(x, x, sc16.float()))

    sd = random_block_state(dim, ffn, heads, seed=2, device=cuda)
    keys = [k for k in sd if k.endswith("norm_q.weight") or k.endswith("norm_k.weight") or k.startswith("norm3.") or k == "modulation"]
    sd16 = {k: (v.bfloat16() if k in keys else v) for k, v in sd.items()}
    sd32 = {k: (v.bfloat16().float() if k in keys else v) for k, v in sd.items()}
    e0 = (torch.randn(6, dim, generator=g) * 0.1).to(cuda)
    ctx = torch.randn(33, dim, generator=g).bfloat16().to(cuda)
    y16 = WanBlockB200(sd16, dim, heads, topk=0.5)(x, e0, ang, ctx)
    y32 = WanBlockB200(sd32, dim, heads, topk=0.5)(x, e0, ang, ctx)
    assert torch.equal(y16, y32)
