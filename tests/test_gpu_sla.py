"""GPU parity for the SLA / SageSLA path (a7-a10) against the CPU oracle and the reference-generated goldens.

Tolerances (the reference states none; SURVEY 8c):
  * block map: bit-exact as a SET, modulo entries whose rounded pooled score ties with the selection threshold;
  * Sage INT8 codes: exact vs the emulation (both IEEE) except where the 16-bit key mean rounds differently;
  * attention output vs the fp32 block-sparse oracle on the same map: cosine >= 0.999, rel-L2 <= 2e-2;
    vs the INT8 emulation oracle: rel-L2 <= 1e-2.
"""
import pytest
import torch

from oracle import golden
from oracle import td_oracle as O

pytestmark = pytest.mark.gpu


def _qkv(b, l, h, d, seed, kbias=2.0, dtype=torch.bfloat16):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(b, l, h, d, generator=g)
    k = torch.randn(b, l, h, d, generator=g) + torch.randn(1, 1, h, d, generator=g) * kbias
    v = torch.randn(b, l, h, d, generator=g)
    return q.to(dtype), k.to(dtype), v.to(dtype)


@pytest.mark.parametrize("b,l,h,d", [(1, 600, 2, 128), (2, 333, 3, 128), (1, 1000, 2, 64), (1, 64, 1, 128)])
def test_quant_qk_pools_and_codes(cuda, b, l, h, d):
    from turbodiffusion_b200.SLA.utils import quant_qk
    q, k, _ = _qkv(b, l, h, d, 100 + l)
    prep = quant_qk(q.to(cuda), k.to(cuda))
    torch.cuda.synchronize()
    qh, kh = q.transpose(1, 2).contiguous(), k.transpose(1, 2).contiguous()
    km_ref = kh.float().mean(-2)
    torch.testing.assert_close(prep.kmean.cpu(), km_ref, rtol=1e-5, atol=1e-5)
    # use the kernel's own (rounded) mean so the remaining comparison is exact arithmetic
    km_t = prep.kmean.cpu().to(q.dtype)[:, :, None, :]
    arg_k = kh - km_t
    assert torch.equal(prep.q_pool.cpu().float(), O.mean_pool(qh, 128).float()) or \
        (prep.q_pool.cpu().float() - O.mean_pool(qh, 128).float()).abs().max() < 2e-2
    pk_ref = O.mean_pool(arg_k, 64)
    assert (prep.k_pool.cpu().float() - pk_ref.float()).abs().max() <= 2.0 ** -7 * pk_ref.float().abs().max() + 1e-6
    q_i8, q_s = O.sage_quant_blocks(qh, 128)
    k_i8, k_s = O.sage_quant_blocks(arg_k, 64)
    assert torch.equal(prep.q_scale.cpu(), q_s) and torch.equal(prep.k_scale.cpu(), k_s)
    assert torch.equal(prep.q_i8.cpu(), q_i8), (prep.q_i8.cpu() != q_i8).sum()
    assert torch.equal(prep.k_i8.cpu(), k_i8), (prep.k_i8.cpu() != k_i8).sum()


def _check_topk_set(scores, sparse_map, lut, topk):
    """Selection is a valid top-k of `scores` (ties free), lut ascending and consistent with the map."""
    assert (sparse_map.sum(-1) == topk).all()
    sel = sparse_map.bool()
    lo = torch.where(sel, scores, torch.full_like(scores, float("inf"))).amin(-1)
    hi = torch.where(~sel, scores, torch.full_like(scores, float("-inf"))).amax(-1)
    assert (lo >= hi).all(), "an unselected block scores higher than a selected one"
    assert (lut[..., 1:] > lut[..., :-1]).all() if topk > 1 else True
    rebuilt = torch.zeros_like(sparse_map)
    rebuilt.scatter_(-1, lut.long(), 1)
    assert torch.equal(rebuilt, sparse_map)


@pytest.mark.parametrize("b,l,h,d,ratio", [(1, 600, 2, 128, 0.25), (2, 333, 3, 128, 0.5), (1, 2100, 2, 128, 0.1),
                                           (1, 1000, 2, 64, 0.15), (1, 600, 1, 128, 1.0)])
def test_block_map_is_an_exact_topk_of_the_rounded_scores(cuda, b, l, h, d, ratio):
    from turbodiffusion_b200.SLA.utils import block_map_from_pools, quant_qk
    q, k, _ = _qkv(b, l, h, d, 7 + l)
    prep = quant_qk(q.to(cuda), k.to(cuda))
    nblk = prep.nblk
    topk = min(nblk, int(ratio * nblk))
    sparse_map, lut = block_map_from_pools(prep.q_pool, prep.k_pool, topk)
    torch.cuda.synchronize()
    # scores recomputed on the CPU from the kernel's own pooled vectors: fp32 dot, rounded to bf16
    scores = (prep.q_pool.cpu().float() @ prep.k_pool.cpu().float().transpose(-1, -2)).to(q.dtype).float()
    sm, lt = sparse_map.cpu(), lut.cpu()
    # accumulation order can move a score by one bf16 ulp; allow the check on a 1-ulp-widened threshold
    try:
        _check_topk_set(scores, sm, lt, topk)
    except AssertionError:
        sel = sm.bool()
        lo = torch.where(sel, scores, torch.full_like(scores, float("inf"))).amin(-1)
        hi = torch.where(~sel, scores, torch.full_like(scores, float("-inf"))).amax(-1)
        bad = hi > lo
        assert ((hi - lo)[bad] <= 2.0 ** -7 * hi[bad].abs() + 1e-6).all()
    # tie rule: among blocks equal to the threshold the lowest indices are taken -> equals the oracle selection
    sm_ref, lut_ref = O.select_topk(scores, topk)
    agree = (sm == sm_ref).float().mean().item()
    assert agree > 0.999, agree


@pytest.mark.parametrize("name", ["sla_a", "sla_b"])
def test_block_map_vs_reference_golden(cuda, name):
    """Golden from the reference's own get_block_map (torch.topk): equal as sets except at threshold ties."""
    from turbodiffusion_b200.SLA.utils import get_block_map
    g = golden.load(name)
    qh = g["q"].transpose(1, 2).contiguous().to(cuda)
    kh = g["k"].transpose(1, 2).contiguous().to(cuda)
    sparse_map, lut, topk = get_block_map(qh, kh, g["topk_ratio"], 128, 64)
    assert topk == g["topk"]
    ours, ref = sparse_map.cpu().bool(), g["sparse_map"].bool()
    diff = ours ^ ref
    if diff.any():
        score = g["score"].float()
        thr = torch.where(ref, score, torch.full_like(score, float("inf"))).amin(-1, keepdim=True)
        near = (score - thr).abs() <= 2.0 ** -6 * thr.abs() + 1e-6
        assert (near | ~diff).all(), "block maps differ away from the selection threshold"
        assert diff.float().mean() < 5e-3


@pytest.mark.parametrize("b,l,h", [(1, 600, 2), (2, 333, 3), (1, 128, 1)])
def test_linear_moments(cuda, b, l, h):
    from turbodiffusion_b200.SLA.core import linear_moments
    d = 128
    _, k, v = _qkv(b, l, h, d, 31 + l)
    kv, ksum = linear_moments(k.to(cuda), v.to(cuda))
    torch.cuda.synchronize()
    kh, vh = k.transpose(1, 2).float(), v.transpose(1, 2).float()
    phi = torch.softmax(kh, -1).to(k.dtype).float()
    kv_ref = vh.transpose(-1, -2) @ phi          # [b,h,dv,dk]
    ks_ref = phi.sum(-2)
    s_kv, s_ks = O.stats(kv.cpu(), kv_ref), O.stats(ksum.cpu(), ks_ref)
    assert s_kv["rel_l2"] < 3e-3 and s_ks["rel_l2"] < 3e-3, (s_kv, s_ks)


CASES = [
    # b, l, h, topk_ratio
    (1, 600, 2, 0.25),    # ragged q tail (600 = 4*128 + 88) and k tail (600 = 9*64 + 24)
    (2, 333, 3, 0.5),
    (1, 1280, 2, 0.1),    # exact multiples
    (1, 700, 1, 1.0),     # dense: every block selected
    (1, 256, 2, 0.3),     # topk = 1 block
]


@pytest.mark.parametrize("b,l,h,ratio", CASES)
def test_sage_sla_forward_vs_oracle(cuda, b, l, h, ratio):
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    from turbodiffusion_b200.SLA.utils import block_map_from_pools, quant_qk
    d = 128
    q, k, v = _qkv(b, l, h, d, 1000 + l)
    g = torch.Generator().manual_seed(5)
    mod = SageSparseLinearAttention(d, ratio).to(cuda)
    with torch.no_grad():
        mod.proj_l.weight.copy_(torch.randn(d, d, generator=g) * 0.05)
        mod.proj_l.bias.copy_(torch.randn(d, generator=g) * 0.05)
    out, sparsity = mod(q.to(cuda), k.to(cuda), v.to(cuda), return_sparsity=True)
    torch.cuda.synchronize()
    assert out.shape == q.shape and out.dtype == q.dtype
    assert not torch.isnan(out.float()).any()
    # oracle on the kernel's own block selection, so this isolates the attention arithmetic
    prep = quant_qk(q.to(cuda), k.to(cuda))
    topk = min(prep.nblk, int(ratio * prep.nblk))
    assert sparsity == topk / prep.nblk
    _, lut = block_map_from_pools(prep.q_pool, prep.k_pool, topk)
    lut = lut.cpu()
    w, bias = mod.proj_l.weight.detach().cpu(), mod.proj_l.bias.detach().cpu()
    exact = O.sla_forward(q, k, v, w, bias, ratio, mode="exact", lut=lut)
    sage = O.sla_forward(q, k, v, w, bias, ratio, mode="sage", lut=lut)
    s_exact, s_sage = O.stats(out.cpu(), exact), O.stats(out.cpu(), sage)
    ref_gap = O.stats(sage, exact)
    assert s_exact["cos"] >= 0.999 and s_exact["rel_l2"] <= 2e-2, (s_exact, ref_gap)
    assert s_sage["rel_l2"] <= 1e-2, (s_sage, ref_gap)


@pytest.mark.parametrize("name", ["sla_a"])
def test_sla_forward_vs_reference_golden(cuda, name):
    """End to end against the output of the reference's SparseLinearAttention.forward (Triton path, CPU interpreter)."""
    from turbodiffusion_b200.SLA import SparseLinearAttention
    g = golden.load(name)
    d = g["q"].shape[-1]
    mod = SparseLinearAttention(d, g["topk_ratio"], BLKQ=128, BLKK=64).to(cuda)
    with torch.no_grad():
        mod.proj_l.weight.copy_(g["proj_w"])
        mod.proj_l.bias.copy_(g["proj_b"])
    out = mod(g["q"].to(cuda), g["k"].to(cuda), g["v"].to(cuda)).cpu()
    s = O.stats(out, g["out"])
    # 128-wide heads: the 16-bit-QK kernel against the reference's Triton path (SURVEY 8c: rel-L2 <= 5e-3 for the bf16 path)
    assert s["cos"] >= 0.9999 and s["rel_l2"] <= 5e-3, s
    # the Sage (INT8-QK) module on the same inputs stays inside its own, wider bound
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    sage = SageSparseLinearAttention(d, g["topk_ratio"]).to(cuda)
    sage.load_state_dict(mod.state_dict())
    s2 = O.stats(sage(g["q"].to(cuda), g["k"].to(cuda), g["v"].to(cuda)).cpu(), g["out"])
    assert s2["cos"] >= 0.999 and s2["rel_l2"] <= 2e-2, s2
    assert s["rel_l2"] < s2["rel_l2"]


@pytest.mark.parametrize("b,l,h,ratio", [(1, 600, 2, 0.25), (2, 333, 3, 0.5), (1, 1280, 2, 0.1), (1, 700, 1, 1.0)])
def test_sla_16bit_qk_forward_vs_oracle(cuda, b, l, h, ratio):
    """SparseLinearAttention (a9'): against the oracle's restatement of the Triton path (P rounded to T, SLA/kernel.py:73) and
    the fp32 oracle, on the kernel's own block selection; ragged tails and the dense case included."""
    from turbodiffusion_b200.SLA import SparseLinearAttention
    d = 128
    q, k, v = _qkv(b, l, h, d, 2000 + l)
    g = torch.Generator().manual_seed(5)
    mod = SparseLinearAttention(d, ratio, BLKQ=128, BLKK=64).to(cuda)
    with torch.no_grad():
        mod.proj_l.weight.copy_(torch.randn(d, d, generator=g) * 0.05)
        mod.proj_l.bias.copy_(torch.randn(d, generator=g) * 0.05)
    out, sel = mod.forward_with_lut(q.to(cuda), k.to(cuda), v.to(cuda))
    torch.cuda.synchronize()
    lut = sel["lut"].cpu()
    w, bias = mod.proj_l.weight.detach().cpu(), mod.proj_l.bias.detach().cpu()
    exact = O.sla_forward(q, k, v, w, bias, ratio, mode="exact", lut=lut)
    tri = O.sla_forward(q, k, v, w, bias, ratio, mode="triton", lut=lut)
    s_exact, s_tri = O.stats(out.cpu(), exact), O.stats(out.cpu(), tri)
    assert s_exact["cos"] >= 0.9999 and s_exact["rel_l2"] <= 5e-3, (s_exact, s_tri)
    assert s_tri["rel_l2"] <= 5e-3, (s_exact, s_tri)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_sage_sla_forward_head_dim_64_and_fp16(cuda, dtype):
    """SageSLA accepts head_dim 64 (SLA/core.py:207) and use_bf16=False (fp16 compute, SLA/core.py:136)."""
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    from turbodiffusion_b200.SLA.utils import block_map_from_pools, quant_qk
    b, l, h, d, ratio = 2, 333, 2, 64, 0.5
    q, k, v = _qkv(b, l, h, d, 77, dtype=dtype)
    g = torch.Generator().manual_seed(5)
    mod = SageSparseLinearAttention(d, ratio, use_bf16=(dtype == torch.bfloat16)).to(cuda)
    with torch.no_grad():
        mod.proj_l.weight.copy_(torch.randn(d, d, generator=g) * 0.05)
        mod.proj_l.bias.copy_(torch.randn(d, generator=g) * 0.05)
    out = mod(q.to(cuda), k.to(cuda), v.to(cuda)).cpu()
    assert out.shape == q.shape and out.dtype == dtype
    import torch.nn.functional as F
    prep = quant_qk(F.pad(q, (0, 64)).to(cuda).contiguous(), F.pad(k, (0, 64)).to(cuda).contiguous())
    topk = min(prep.nblk, int(ratio * prep.nblk))
    _, lut = block_map_from_pools(prep.q_pool, prep.k_pool, topk)
    w, bias = mod.proj_l.weight.detach().cpu(), mod.proj_l.bias.detach().cpu()
    exact = O.sla_forward(q, k, v, w, bias, ratio, mode="exact", lut=lut.cpu(), dtype=dtype)
    s = O.stats(out, exact)
    assert s["cos"] >= 0.999 and s["rel_l2"] <= 2e-2, s


def test_sla_forward_vs_reference_golden_d64(cuda):
    from turbodiffusion_b200.SLA import SparseLinearAttention
    g = golden.load("sla_b")
    mod = SparseLinearAttention(64, g["topk_ratio"], BLKQ=128, BLKK=64).to(cuda)
    with torch.no_grad():
        mod.proj_l.weight.copy_(g["proj_w"])
        mod.proj_l.bias.copy_(g["proj_b"])
    out = mod(g["q"].to(cuda), g["k"].to(cuda), g["v"].to(cuda)).cpu()
    s = O.stats(out, g["out"])
    assert s["cos"] >= 0.999 and s["rel_l2"] <= 2e-2, s


def test_fp16_block_map_and_quant(cuda):
    from turbodiffusion_b200.SLA.utils import quant_qk
    q, k, _ = _qkv(1, 600, 2, 128, 3, dtype=torch.float16)
    prep = quant_qk(q.to(cuda), k.to(cuda))
    qh = q.transpose(1, 2).contiguous()
    q_i8, q_s = O.sage_quant_blocks(qh, 128)
    assert torch.equal(prep.q_scale.cpu(), q_s) and torch.equal(prep.q_i8.cpu(), q_i8)


@pytest.mark.parametrize("pattern,qscale,l,h,ratio", [
    ("all", 8.0, 1280, 2, 0.5),          # every row's running maximum jumps by > 2^8 somewhere
    ("all", 16.0, 700, 1, 1.0),          # dense selection, ragged q tail (60 rows) and k tail (60 keys)
    ("half_warp", 16.0, 640, 2, 1.0),    # rows 0-15 of every 32-row group are scaled: each warp takes the branch for half its rows
    ("one_warp", 16.0, 640, 2, 1.0),     # only rows 0-31 of every query block (softmax warp 0) are scaled
    ("ragged_last", 12.0, 1000, 2, 1.0), # the maximum of many rows sits in the ragged LAST key block (40 valid keys)
])
def test_sage_sla_forward_large_scores_exercise_the_lazy_rescale(cuda, pattern, qscale, l, h, ratio):
    """With unit-variance q,k the per-block row maxima differ by far less than the lazy-rescale threshold (2^8), so ordinary
    cases never take the branch that rescales the O accumulator in tensor memory.  Scaling q makes the log2-domain scores
    spread over tens of units: the running maximum grows by more than 8 between key blocks.  Patterns cover a branch taken
    by all rows, by part of a warp (alpha = 1 for the other rows), by one warp of the CTA only, and a rescale triggered by
    the ragged last key block.  Compared against the INT8 emulation (same score quantisation) and the fp32 oracle."""
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    from turbodiffusion_b200.SLA.utils import block_map_from_pools, quant_qk
    d = 128
    q, k, v = _qkv(1, l, h, d, 4000 + l)
    qf = q.float()
    rows = torch.arange(l)
    if pattern == "all" or pattern == "ragged_last":
        qf = qf * qscale
    elif pattern == "half_warp":
        qf[:, (rows % 32) < 16] *= qscale
    elif pattern == "one_warp":
        qf[:, (rows % 128) < 32] *= qscale
    if pattern == "ragged_last":
        # every query gets a common component along u and the keys of the last (ragged) block point along u, so the row
        # maximum of most rows sits in that block and exceeds everything seen before by more than 2^8
        nlast = l - (l // 64) * 64
        u = torch.ones(d) / d ** 0.5
        qf = qf + 2.0 * qscale * u
        kf = k.float()
        kf[:, -nlast:] += 6.0 * u
        k = kf.bfloat16()
    q = qf.bfloat16()
    g = torch.Generator().manual_seed(6)
    mod = SageSparseLinearAttention(d, ratio).to(cuda)
    with torch.no_grad():
        mod.proj_l.weight.copy_(torch.randn(d, d, generator=g) * 0.05)
        mod.proj_l.bias.copy_(torch.randn(d, generator=g) * 0.05)
    out, sel = mod.forward_with_lut(q.to(cuda), k.to(cuda), v.to(cuda))
    torch.cuda.synchronize()
    assert not torch.isnan(out.float()).any() and not torch.isinf(out.float()).any()
    lut = sel["lut"].cpu()
    w, bias = mod.proj_l.weight.detach().cpu(), mod.proj_l.bias.detach().cpu()
    # how often the branch is taken according to the oracle's scores: rows whose running max grows by > 8 (log2 units)
    qh, kh = q.transpose(1, 2).float(), k.transpose(1, 2).float()
    s = (qh @ (kh - kh.mean(-2, keepdim=True)).transpose(-1, -2)) * (d ** -0.5) * 1.4426950408889634
    blk_max = torch.stack([s[..., i:i + 64].amax(-1) for i in range(0, l, 64)], -1)        # [1,h,l,nblk] (dense order)
    run_max = torch.cummax(blk_max, -1).values
    grows = (run_max[..., 1:] - run_max[..., :-1]) > 8
    frac = grows.any(-1).float().mean().item()
    assert frac > (0.3 if pattern in ("all", "ragged_last") else 0.08), frac
    if pattern == "ragged_last":
        assert grows[..., -1].float().mean() > 0.2, "the ragged last block should trigger the rescale for many rows"
    sage = O.sla_forward(q, k, v, w, bias, ratio, mode="sage", lut=lut)
    exact = O.sla_forward(q, k, v, w, bias, ratio, mode="exact", lut=lut)
    s_sage, s_exact = O.stats(out.cpu(), sage), O.stats(out.cpu(), exact)
    assert s_sage["rel_l2"] <= 3e-2, (s_sage, s_exact)       # the emulation itself is 4-5e-2 away from fp32 on these inputs
    assert s_exact["cos"] >= 0.99, (s_sage, s_exact)


@pytest.mark.parametrize("feature_map,d,l,h,ratio", [("elu", 128, 600, 2, 0.25), ("relu", 128, 333, 3, 0.5), ("softmax", 64, 1000, 3, 0.15),
                                                     ("elu", 64, 700, 2, 0.3)])
def test_sla_feature_maps_and_native_64_wide_heads(cuda, feature_map, d, l, h, ratio):
    """SLA/core.py:57-73 feature maps (elu+1, relu) of the linear branch and 64-wide heads (SLA/core.py:207) on the native
    tiles (odd head counts exercise the unpaired head of the moments kernel).  Oracle: fp32 block-sparse attention + fp32
    linear branch with the same feature map on the kernel's own block selection."""
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    q, k, v = _qkv(1, l, h, d, 6000 + l + d)
    q = (q.float() * 0.5).bfloat16()          # keep elu/relu features in a range where the linear branch matters
    g = torch.Generator().manual_seed(8)
    mod = SageSparseLinearAttention(d, ratio, feature_map=feature_map).to(cuda)
    with torch.no_grad():
        mod.proj_l.weight.copy_(torch.randn(d, d, generator=g) * 0.05)
        mod.proj_l.bias.copy_(torch.randn(d, generator=g) * 0.05)
    out, sel = mod.forward_with_lut(q.to(cuda), k.to(cuda), v.to(cuda))
    torch.cuda.synchronize()
    lut = sel["lut"].cpu()
    w, b = mod.proj_l.weight.detach().cpu(), mod.proj_l.bias.detach().cpu()
    mblk = (l + 127) // 128
    worst = 0.0
    for head in range(h):
        for m in range(mblk):
            ref = O.sla_forward_block(q, k, v, w, b, head, m, lut[0, head, m], mode="exact", feature_map=feature_map)
            got = out[0, m * 128:min(l, (m + 1) * 128), head].cpu()
            s = O.stats(got, ref)
            assert s["cos"] >= 0.999 and s["rel_l2"] <= 2e-2, (feature_map, d, head, m, s)
            worst = max(worst, s["rel_l2"])
    print("feature map", feature_map, d, "worst rel_l2", worst)


@pytest.mark.parametrize("d,h,feature", [(64, 3, 0), (64, 4, 1), (128, 2, 2)])
def test_linear_moments_head_dims_and_feature_maps(cuda, d, h, feature):
    from turbodiffusion_b200.SLA.core import linear_moments
    l = 700
    _, k, v = _qkv(1, l, h, d, 90 + d + h)
    kv, ksum = linear_moments(k.to(cuda), v.to(cuda), feature)
    torch.cuda.synchronize()
    fq, fk = O.feature_maps(["softmax", "elu", "relu"][feature])
    kh, vh = k.transpose(1, 2).float(), v.transpose(1, 2).float()
    phi = fk(kh).to(k.dtype).float()
    kv_ref = vh.transpose(-1, -2) @ phi
    s_kv, s_ks = O.stats(kv.cpu(), kv_ref), O.stats(ksum.cpu(), phi.sum(-2))
    assert s_kv["rel_l2"] < 3e-3 and s_ks["rel_l2"] < 3e-3, (s_kv, s_ks)


def test_ltx_sparse_only_call_sequence(cuda):
    """The call sequence of TurboT2AV's LTXSageSLAAttention._sparse_only_forward (ltx_distillation/acceleration.py:260-383)
    against the names it looks up in SLA.core; with proj_l == 0 it must equal SageSparseLinearAttention.forward."""
    import turbodiffusion_b200.SLA.core as sla_core
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    b, l, h, d, topk = 1, 900, 2, 128, 0.3
    q, k, v = (t.to(cuda) for t in _qkv(b, l, h, d, 321))
    mod = SageSparseLinearAttention(d, topk).to(cuda)          # proj_l zero-initialised (SLA/core.py:163-166)
    want = mod(q, k, v)
    qh, kh, vh = (t.transpose(1, 2).contiguous() for t in (q, k, v))
    assert sla_core.get_cuda_arch(0) == "sm100"
    sparse_map, _, _ = sla_core.get_block_map(qh, kh, topk_ratio=topk, BLKQ=128, BLKK=64)
    km = kh.mean(dim=-2, keepdim=True)
    q_int8, q_scale, k_int8, k_scale = sla_core.get_vanilla_qk_quant(qh, kh, km, 128, 64)
    lut, valid_block_num = sla_core.block_map_lut_triton(sparse_map)
    assert (valid_block_num == int(topk * ((l + 63) // 64))).all()
    o_s = torch.empty_like(qh)
    padded = (l + 127) // 128 * 128
    v_t = torch.empty((b, h, d, padded), dtype=vh.dtype, device=cuda)
    sla_core.fused.transpose_pad_permute_cuda(vh, v_t, 1)
    v_fp8 = torch.empty(v_t.shape, dtype=torch.float8_e4m3fn, device=cuda)
    v_scale = torch.empty((b, h, d), dtype=torch.float32, device=cuda)
    sla_core.fused.scale_fuse_quant_cuda(v_t, v_fp8, v_scale, l, 2.25, 1)
    pv = torch.full((h,), 1e6, dtype=torch.float32, device=cuda)
    assert sla_core.SAGE2PP_ENABLED
    sla_core.qk_int8_sv_f8_accum_f16_block_sparse_attn_inst_buf_fuse_v_scale_with_pv_threshold(
        q_int8, k_int8, v_fp8, o_s, lut, valid_block_num, pv, q_scale, k_scale, v_scale, 1, False, 1, 1.0 / d ** 0.5, 0)
    got = o_s.transpose(1, 2)
    assert torch.equal(got.contiguous(), want)
    # a map that did not come from get_block_map is rebuilt from its entries
    lut2, _ = sla_core.block_map_lut_triton(sparse_map.clone())
    assert torch.equal(lut2, lut)
    with pytest.raises(NotImplementedError):
        sla_core.qattn.qk_int8_sv_f16_accum_f16_block_sparse_attn_inst_buf_with_pv_threshold


def test_mean_pool_block_sizes(cuda):
    from turbodiffusion_b200.SLA.utils import mean_pool
    x = _qkv(1, 700, 2, 128, 55)[1].transpose(1, 2).contiguous()
    for blk in (64, 128):
        got = mean_pool(x.to(cuda), blk).cpu()
        ref = O.mean_pool(x, blk)
        assert (got.float() - ref.float()).abs().max() <= 2.0 ** -6 * ref.float().abs().max()


@pytest.mark.parametrize("l,h,d,shards", [(1000, 3, 128, (384, 384, 232)), (690, 2, 128, (384, 306)), (1000, 2, 64, (512, 488))])
def test_split_key_prep_equals_the_fused_one(cuda, l, h, d, shards):
    """The sequence-parallel form of the key half (dist.py): per-shard 128-row partial sums -> concatenated -> kmean_final, then
    each shard quantised on its own with the INT8 codes left in the [B, L, H, D] layout, reproduces tdb200_sla_quant_qk's
    key mean, codes, scales and pooled means BIT FOR BIT (shard boundaries are multiples of 128 rows)."""
    from turbodiffusion_b200.SLA.utils import QKPrep, kmean_from_partials, kmean_partials, quant_k_into, quant_k_seq
    assert sum(shards) == l
    _, k, _ = _qkv(1, l, h, d, seed=31)
    k = k.to(cuda)
    ref = quant_k_into(QKPrep(), k, l)
    parts, row = [], 0
    for n in shards:
        parts.append(kmean_partials(k[:, row:row + n].contiguous()))
        row += n
    partials = torch.cat(parts, dim=2).contiguous()
    assert partials.shape[2] == (l + 127) // 128
    kmean = kmean_from_partials(partials, l)
    assert torch.equal(kmean, ref.kmean)
    codes, scales, pools, row = [], [], [], 0
    for n in shards:
        c, s, p = quant_k_seq(k[:, row:row + n].contiguous(), kmean)
        assert c.shape == (1, n, h, d)
        codes.append(c), scales.append(s), pools.append(p)
        row += n
    assert torch.equal(torch.cat(codes, 1).transpose(1, 2), ref.k_i8)
    assert torch.equal(torch.cat(scales, 2), ref.k_scale)
    assert torch.equal(torch.cat(pools, 2), ref.k_pool)


def test_attention_reads_sequence_major_int8_keys(cuda):
    """tdb200_sla_attn_fwd_kseq (INT8 K in the gathered [B, Lk, H, D] layout, key rows padded past lk) == tdb200_sla_attn_fwd."""
    from turbodiffusion_b200.SLA.core import attn_fwd, linear_moments
    from turbodiffusion_b200.SLA.utils import block_map_from_pools, quant_qk
    b, l, h, d = 1, 1000, 3, 128
    q, k, v = (t.to(cuda) for t in _qkv(b, l, h, d, seed=32))
    prep = quant_qk(q, k)
    topk = 5
    _, lut = block_map_from_pools(prep.q_pool, prep.k_pool, topk)
    kv, ksum = linear_moments(k, v)
    g = torch.Generator().manual_seed(3)
    w = (torch.randn(d, d, generator=g) * 0.05).to(cuda)
    pb = (torch.randn(d, generator=g) * 0.05).to(cuda)
    kvw = torch.matmul(w, kv).to(q.dtype).contiguous()
    ref = attn_fwd(prep, v, q, lut, topk, kvw, ksum, pb, d ** -0.5)
    pad = 152                                                  # the gathered slab carries zero rows past lk
    k_seq = torch.zeros(b, l + pad, h, d, dtype=torch.int8, device=cuda)
    k_seq[:, :l] = prep.k_i8.transpose(1, 2)
    v_pad = torch.zeros(b, l + pad, h, d, dtype=v.dtype, device=cuda)
    v_pad[:, :l] = v
    prep.k_i8, prep.k_seq_major = k_seq, True
    got = attn_fwd(prep, v_pad, q, lut, topk, kvw, ksum, pb, d ** -0.5, lk=l)
    assert torch.equal(got, ref)


@pytest.mark.parametrize("d,h,dtype", [(128, 3, torch.bfloat16), (64, 4, torch.float16)])
def test_project_moments_equals_the_matmul(cuda, d, h, dtype):
    """kvw = T(proj_w . kv) (one launch) against torch.matmul in fp32 + cast: same values up to the summation order of the fp32
    chain (a last-place flip of the 16-bit result on a few elements)."""
    from turbodiffusion_b200.SLA.core import project_moments
    g = torch.Generator().manual_seed(d + h)
    w = (torch.randn(d, d, generator=g) * 0.05).to(cuda)
    kv = (torch.randn(2, h, d, d, generator=g) * 3).to(cuda)
    got = project_moments(w, kv, dtype)
    ref = torch.matmul(w.double(), kv.double())
    assert got.shape == (2, h, d, d) and got.dtype == dtype
    err = (got.double() - ref).abs()
    ulp = ref.abs().clamp_min(1e-3) * (2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -11)
    assert (err <= ulp).all(), (err / ulp).max().item()     # within one rounding of T of the exact product
