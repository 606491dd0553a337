"""Pin the CPU oracle against outputs of the REFERENCE's own code (tests/golden/*.pt, produced by
tools/make_golden.py with the reference's Triton kernels run through Triton's CPU interpreter)."""
import os

import pytest
import torch

from oracle import golden
from oracle import td_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    return golden.load(name)


def _max_ulp(got, ref):
    g, r = got.float(), ref.float()
    ulp = torch.maximum(r.abs(), torch.tensor(1e-30)).log2().floor().exp2() * 2.0 ** -7
    return ((g - r).abs() / ulp).max().item(), (g != r).float().mean().item()


@pytest.mark.parametrize("n", [1536, 5120, 256])
def test_fast_norms_match_reference_triton_kernels(n):
    g = _load(f"norm_n{n}")
    x, w, b, eps = g["x"], g["w"], g["b"], g["eps"]
    for got, ref in ((O.fast_rmsnorm(x, w, eps), g["rms"]), (O.fast_layernorm(x, None, None, eps), g["ln"]),
                     (O.fast_layernorm(x, w, b, eps), g["ln_aff"])):
        worst, frac = _max_ulp(got, ref)
        assert worst <= 1.0 and frac < 5e-3, (worst, frac)
    torch.testing.assert_close(O.layernorm_f32(x, None, None, eps), g["ln_f32"], rtol=2e-5, atol=2e-5)


@pytest.mark.parametrize("n", [1536, 5120])
def test_reference_layernorm_really_has_the_padding_term(n):
    """The golden (reference Triton kernel) is reproduced WITH the (N2-N)*mean^2 term and not without it."""
    g = _load(f"norm_n{n}")
    with_q = (O.layernorm_f32(g["x"], None, None, g["eps"], True) - g["ln_f32"]).abs().max().item()
    without = (O.layernorm_f32(g["x"], None, None, g["eps"], False) - g["ln_f32"]).abs().max().item()
    assert with_q < 1e-5 and without > 20 * with_q, (with_q, without)


@pytest.mark.parametrize("name", ["sla_a", "sla_b"])
def test_block_map_pipeline_matches_reference(name):
    g = _load(name)
    qh, kh = g["q"].transpose(1, 2).contiguous(), g["k"].transpose(1, 2).contiguous()
    arg_k, _ = O.smooth_k(kh)
    for got, ref in ((O.mean_pool(qh, 128), g["pooled_q"]), (O.mean_pool(arg_k, 64), g["pooled_k"])):
        worst, frac = _max_ulp(got, ref)
        assert worst <= 1.0 and frac < 2e-3, (worst, frac)
    score = O.pooled_scores(qh, kh, 128, 64)
    worst, frac = _max_ulp(score, g["score"])
    assert worst <= 1.0 and frac < 5e-3, (worst, frac)
    # selection: equal as a set to torch.topk's, except where the score ties with the threshold
    sm, lut, topk = O.get_block_map(qh, kh, g["topk_ratio"], 128, 64)
    assert topk == g["topk"]
    sm_ref = g["sparse_map"].bool()
    diff = sm.bool() ^ sm_ref
    if diff.any():
        sc = g["score"].float()
        thr = torch.where(sm_ref, sc, torch.full_like(sc, float("inf"))).amin(-1, keepdim=True)
        assert ((sc - thr).abs() <= 2.0 ** -6 * thr.abs() + 1e-6)[diff].all()
    # the ascending LUT is the sorted version of the reference's unsorted index list
    if not diff.any():
        assert torch.equal(lut.long(), torch.sort(g["lut"], -1).values)


@pytest.mark.parametrize("name", ["sla_a", "sla_b"])
def test_sparse_attention_and_module_match_reference(name):
    g = _load(name)
    qh, kh, vh = (g[t].transpose(1, 2).contiguous() for t in ("q", "k", "v"))
    lut = torch.sort(g["lut"], -1).values
    o_s = O.sparse_attention(qh, kh, vh, lut, 128, 64, p_dtype=torch.bfloat16).to(torch.bfloat16)
    s = O.stats(o_s, g["o_s"])
    assert s["rel_l2"] < 3e-3, s      # bf16 output rounding + summation order only
    exact = O.sparse_attention(qh, kh, vh, lut, 128, 64)
    assert O.stats(exact, g["o_s"])["rel_l2"] < 5e-3
    out = O.sla_forward(g["q"], g["k"], g["v"], g["proj_w"], g["proj_b"], g["topk_ratio"], mode="triton", lut=lut)
    s = O.stats(out, g["out"])
    assert s["rel_l2"] < 4e-3, s
    out_exact = O.sla_forward(g["q"], g["k"], g["v"], g["proj_w"], g["proj_b"], g["topk_ratio"], mode="exact", lut=lut)
    s = O.stats(out_exact, g["out"])
    assert s["rel_l2"] < 1e-2, s
    # the INT8 emulation stays within the stated Sage tolerance of the reference bf16 path
    out_sage = O.sla_forward(g["q"], g["k"], g["v"], g["proj_w"], g["proj_b"], g["topk_ratio"], mode="sage", lut=lut)
    s = O.stats(out_sage, g["out"])
    assert s["cos"] > 0.999 and s["rel_l2"] < 2e-2, s


def test_ltx_modulation_known_answers():
    """Formulas pinned by the reference's only known-answer tests for the prologue math
    (TurboT2AV/LTX-2/packages/ltx-core/tests/test_transformer_fusion_helpers.py:13-87): rms(x)*(1+scale)+shift etc."""
    torch.manual_seed(7)
    x = torch.randn(2, 3, 4)
    table = torch.randn(6, 4)
    timestep = torch.randn(2, 3, 24)
    ada = table[None, None] + timestep.view(2, 3, 6, 4)
    shift, scale, gate = ada[:, :, 0], ada[:, :, 1], ada[:, :, 2]
    expected = O.ltx_rms_norm(x) * (1 + scale) + shift
    manual = x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + 1e-6) * (1 + scale) + shift
    torch.testing.assert_close(expected, manual)
    res = torch.randn(2, 3, 4)
    torch.testing.assert_close(x + res * gate, O.gate_residual(x, res, gate[0, 0]) if False else x + res * gate)


def test_int8_quant_known_values():
    x = torch.zeros(128, 128, dtype=torch.bfloat16)
    x[0, 0], x[0, 1], x[1, 0] = 4.0, -4.0, 0.0157
    q, s = O.int8_quant(x)
    assert s.shape == (1, 1) and s[0, 0].item() == 4.0 / 128
    assert q[0, 0].item() == 127 and q[0, 1].item() == -128   # +128 saturates to 127, -128 is representable
    assert q[1, 0].item() == round(float(torch.tensor(0.0157).bfloat16()) * 32)


def test_c_and_torch_gemm_oracles_agree():
    torch.manual_seed(0)
    x, w = torch.randn(200, 384).bfloat16(), (torch.randn(136, 384) * 0.05).bfloat16()
    a_q, a_s = O.int8_quant(x)
    b_q, b_s = O.int8_quant(w)
    y1 = O.int8_gemm_f32(a_q, a_s, b_q, b_s)
    y2 = O._int8_gemm_f32_torch(a_q, a_s, b_q, b_s)
    assert torch.equal(y1, y2)
    s = O.stats(y1, x.float() @ w.float().t())
    assert s["rel_l2"] < 2e-2


def test_dense_sdpa_equals_sparse_with_all_blocks():
    torch.manual_seed(1)
    q, k, v = (torch.randn(1, 2, 200, 64).bfloat16() for _ in range(3))
    lut = torch.arange(4).view(1, 1, 1, 4).expand(1, 2, 2, 4)
    sp = O.sparse_attention(q, k, v, lut, 128, 64)
    de = O.dense_attention(q.float(), k.float(), v.float())
    assert O.stats(sp, de)["rel_l2"] < 1e-5


@pytest.mark.parametrize("k", [384, 4096])
def test_ltx_row_quant_matches_the_reference_triton_kernel(k):
    """oracle.ltx_row_quant_int8 against the reference's own `_row_quant_kernel` (tilelang_w8a8.py:16-36) executed through
    Triton's CPU interpreter (tools/make_golden.py ltx): zero row (1e-4 floor), exact .5 ties, outlier columns."""
    g = torch.load(os.path.join(GOLD, f"ltx_rowquant_k{k}.pt"))
    q, s = O.ltx_row_quant_int8(g["x"])
    assert torch.equal(s, g["s"]) and torch.equal(q, g["q"])
    assert g["q"][5, :8].tolist() == [127, 64, -64, 1, -1, 2, -2, 3]          # round half away from zero
    assert g["s"][3].item() == pytest.approx(1e-4 / 127.0, rel=1e-6)


def test_ltx_post_scale_epilogue_is_a_fused_multiply_add():
    """The reference's TileLang epilogue executes fma(float(acc)*sA, sB, bias) (tools/tilelang_epilogue_probe.py,
    profiles/r01_tilelang_epilogue_sass.txt).  Known answer where the fused and the unfused evaluation differ:
    (1+2^-12)(1+3*2^-12) = 1 + 2^-10 + 3*2^-24 is a rounding tie for a separate multiply (-> 1 + 2^-10 + 2^-22); with
    bias = -(1+2^-10) the unfused result is 4*2^-24, the fused one keeps 3*2^-24."""
    a_q = torch.tensor([[1] + [0] * 127], dtype=torch.int8)
    b_q = torch.tensor([[1] + [0] * 127], dtype=torch.int8)
    a_s = torch.tensor([1.0 + 2.0 ** -12])
    b_s = torch.tensor([1.0 + 3 * 2.0 ** -12])
    bias = torch.tensor([-(1.0 + 2.0 ** -10)]).half()
    y = O.ltx_gemm_post_scale(a_q, a_s, b_q, b_s, bias, out_dtype=torch.float32)
    assert y.item() == 3 * 2.0 ** -24
    assert ((a_s * b_s) + bias.float()).item() == 4 * 2.0 ** -24      # what an unfused mul + add would return
