"""Run-to-run reproducibility and completeness of every kernel, and of the denoise step at the real Wan-1.3B width.

(a) Every non-diagnostic entry point of include/tdb200.h is called twice through the C ABI on identical inputs, with every
    output and workspace filled with 0xFF before the first run and with 0x00 before the second.  Equal bytes across the two
    runs mean no element is left unwritten and nothing depends on scheduling; a guard tail behind every buffer must keep
    its poison (no write past a ragged last tile).  Accumulating outputs (kv, ksum) are prefilled with the same non-zero
    values in both runs instead and must equal prefill + the zero-prefill result.
(b) WanHotPath.step: two eager steps, the CUDA-graph replay (captured the way bench.py captures it) and the blocks chained
    without the LayerNorm-statistics / modulation-table fusions are all bit-identical.
(c) Every layer of that step against the CPU oracle, fed the GPU's input and the kernel's own block selection.
(d) The W8A8 GEMM bit for bit at the real K and N of Wan-1.3B / 14B (K loops of 70-108 blocks, up to ~32k tiles).
"""
import math

import pytest
import torch

from oracle import td_oracle as O

GUARD = 4096   # bytes of poison behind every output buffer
POISON = (0xFF, 0x00)


def _buffers(specs, fill, device):
    raw, views = {}, {}
    for name, (shape, dtype, _) in specs.items():
        n = math.prod(shape) * torch.empty((), dtype=dtype).element_size()
        raw[name] = torch.full((n + GUARD,), fill, dtype=torch.uint8, device=device)
        views[name] = raw[name][:n].view(dtype).view(shape)
    return raw, views


def check_rerun_with_poison(specs, call, device, prefill=None):
    """specs: name -> (shape, dtype, role), role "out" (compared), "ws" (scratch: poisoned, guarded, not compared) or "acc"
    (accumulated into: prefilled from `prefill[name]` in every run).  call(views) runs the kernel.  Returns the first run's
    outputs."""
    prefill = prefill or {}
    runs = []
    for fill in POISON:
        raw, views = _buffers(specs, fill, device)
        for name, t in prefill.items():
            views[name].copy_(t)
        call(views)
        if torch.device(device).type == "cuda":
            torch.cuda.synchronize(device)
        for name, r in raw.items():
            bad = (r[-GUARD:] != fill).nonzero()
            assert bad.numel() == 0, f"{name}: {bad.numel()} guard bytes overwritten, first at byte +{bad[0].item()} past the end"
        runs.append((raw, views))
    for name, (shape, dtype, role) in specs.items():
        if role == "ws":
            continue
        a, b = runs[0][0][name][:-GUARD], runs[1][0][name][:-GUARD]
        diff = (a != b).nonzero()
        assert diff.numel() == 0, (f"{name} {tuple(shape)} {dtype}: {diff.numel()} of {a.numel()} bytes differ between the "
                                   f"0xFF- and the 0x00-poisoned run (never written, or run-dependent); first byte "
                                   f"{diff[0].item()}")
    return {n: v.clone() for n, v in runs[0][1].items()}


# ---- the helper itself (CPU) -----------------------------------------------------------------------------------------
def test_poison_helper_reports_an_unwritten_row():
    x = torch.randn(37, 24)
    full = {"y": ((37, 24), torch.float32, "out")}
    check_rerun_with_poison(full, lambda o: o["y"].copy_(x * 2), "cpu")

    def skips_last_row(o):
        o["y"][:-1].copy_(x[:-1] * 2)
    with pytest.raises(AssertionError, match="differ between"):
        check_rerun_with_poison(full, skips_last_row, "cpu")


def test_poison_helper_reports_a_write_past_the_end():
    def overruns(o):
        o["y"].copy_(torch.ones(10))
        whole = torch.empty(0, dtype=torch.uint8).set_(o["y"].untyped_storage(), 0, (48,))
        whole[40:48] = 7                                                   # 8 bytes beyond the 10 floats
    with pytest.raises(AssertionError, match="guard bytes"):
        check_rerun_with_poison({"y": ((10,), torch.float32, "out")}, overruns, "cpu")


def test_poison_helper_reports_run_dependent_results():
    runs = iter(range(2))
    with pytest.raises(AssertionError, match="differ between"):
        check_rerun_with_poison({"y": ((4,), torch.int32, "out")}, lambda o: o["y"].fill_(next(runs)), "cpu")


# ---- (a) every entry point through the C ABI -----------------------------------------------------------------------------
SIZES = {
    # m rows / dim / ffn of the row kernels and GEMMs; SLA (b, l, h, d); LTX (b, tokens, n)
    "small": dict(m=300, n=384, k=640, ffn=768, sla=(2, 300, 3, 128), ltx=(2, 77, 512)),
    "A": dict(m=32760, n=1536, k=1536, ffn=8960, sla=(1, 32760, 12, 128), ltx=(1, 28672, 4096)),
}


def _cases(sz, dev):
    """name -> builder() returning (specs, call[, prefill]); inputs are made by the builder, on `dev`."""
    from turbodiffusion_b200 import _lib
    from turbodiffusion_b200.SLA.core import linear_moments, moments_workspace_bytes, project_moments
    from turbodiffusion_b200.SLA.utils import block_map_from_pools, quant_k_seq, quant_qk

    lib = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(11)
    bf, f32, i8, i32 = torch.bfloat16, torch.float32, torch.int8, torch.int32
    BF = _lib.DTYPE_TAG[bf]
    P = _lib.ptr

    def S():
        return _lib.stream_ptr(dev)

    def rnd(*shape, scale=1.0, dtype=bf):
        return (torch.randn(*shape, device=dev, generator=g) * scale).to(dtype)

    def ok(rc):
        assert rc == 0, lib.tdb200_last_error()

    def cdiv(a, b):
        return (a + b - 1) // b

    m, n, k, ffn = sz["m"], sz["n"], sz["k"], sz["ffn"]
    eps = 1e-6
    x16 = rnd(m, n)
    cases = {}

    def quant_inputs(rows, cols, seed_scale=0.01):
        q = torch.randint(-128, 128, (rows, cols), device=dev, generator=g, dtype=i8)
        s = torch.rand(cdiv(rows, 128), cols // 128, device=dev, generator=g) * seed_scale + 1e-4
        return q, s

    a_q, a_s = quant_inputs(m, k)
    b_q, b_s = quant_inputs(ffn, k)
    bias = rnd(ffn, scale=0.1)

    # a1 quantisation
    for fn in ("tdb200_quant_int8_block128", "tdb200_gelu_quant_int8_block128"):
        cases[fn] = lambda fn=fn: ({"q": ((m, n), i8, "out"), "s": ((cdiv(m, 128), cdiv(n, 128)), f32, "out")},
                                   lambda o: ok(getattr(lib, fn)(P(x16), BF, m, n, P(o["q"]), P(o["s"]), S())))
    # a2 GEMMs
    cases["tdb200_gemm_w8a8"] = lambda: ({"c": ((m, ffn), bf, "out")}, lambda o: ok(lib.tdb200_gemm_w8a8(
        P(a_q), P(a_s), P(b_q), P(b_s), P(bias), P(o["c"]), BF, m, ffn, k, S())))
    cases["tdb200_gemm_w8a8_ex"] = lambda: ({"c": ((m, ffn), bf, "out")}, lambda o: ok(lib.tdb200_gemm_w8a8_ex(
        P(a_q), P(a_s), P(b_q), P(b_s), P(bias), P(o["c"]), BF, m, ffn, k, 1, S())))
    n3 = 3 * 256 if m < 1000 else 3 * n
    w3_q, w3_s = quant_inputs(n3, k)
    b3 = rnd(n3, scale=0.1)
    cases["tdb200_gemm_w8a8_split"] = lambda: ({"c": ((3, m, n3 // 3), bf, "out")}, lambda o: ok(lib.tdb200_gemm_w8a8_split(
        P(a_q), P(a_s), P(w3_q), P(w3_s), P(b3), P(o["c"]), BF, m, n3, k, 3, S())))
    cases["tdb200_gemm_w8a8_quant_out"] = lambda: (
        {"q": ((m, ffn), i8, "out"), "s": ((cdiv(m, 128), ffn // 128), f32, "out")},
        lambda o: ok(lib.tdb200_gemm_w8a8_quant_out(P(a_q), P(a_s), P(b_q), P(b_s), P(bias), P(o["q"]), P(o["s"]), BF, m, ffn,
                                                    k, 1, S())))
    # a3/a4 norms
    x32 = x16.float()
    w, bb = torch.rand(n, device=dev, generator=g) + 0.5, rnd(n, scale=0.1, dtype=f32)
    sc, sh = rnd(n, scale=0.1, dtype=f32), rnd(n, scale=0.1, dtype=f32)
    cases["tdb200_rms_norm_f32"] = lambda: ({"y": ((m, n), f32, "out")}, lambda o: ok(lib.tdb200_rms_norm_f32(
        P(x32), P(w), P(o["y"]), m, n, eps, S())))
    cases["tdb200_layer_norm_f32"] = lambda: ({"y": ((m, n), f32, "out")}, lambda o: ok(lib.tdb200_layer_norm_f32(
        P(x32), P(w), P(bb), P(o["y"]), m, n, eps, S())))
    cases["tdb200_rms_norm"] = lambda: ({"y": ((m, n), bf, "out")}, lambda o: ok(lib.tdb200_rms_norm(
        P(x16), BF, P(w), P(o["y"]), m, n, eps, S())))
    cases["tdb200_layer_norm"] = lambda: ({"y": ((m, n), bf, "out")}, lambda o: ok(lib.tdb200_layer_norm(
        P(x16), BF, P(w), P(bb), P(o["y"]), m, n, eps, S())))
    # a5 AdaLN
    cases["tdb200_layer_norm_modulate"] = lambda: ({"y": ((m, n), bf, "out")}, lambda o: ok(lib.tdb200_layer_norm_modulate(
        P(x16), BF, P(sc), P(sh), P(o["y"]), m, n, eps, S())))
    quant_specs = {"q": ((m, n), i8, "out"), "s": ((cdiv(m, 128), cdiv(n, 128)), f32, "out")}
    cases["tdb200_layer_norm_modulate_quant"] = lambda: (
        dict(quant_specs, row_stats=((2 * m,), f32, "ws")),
        lambda o: ok(lib.tdb200_layer_norm_modulate_quant(P(x16), BF, P(sc), P(sh), P(o["q"]), P(o["s"]), P(o["row_stats"]),
                                                          m, n, eps, S())))
    y16 = rnd(m, n)
    cases["tdb200_gate_residual"] = lambda: ({"out": ((m, n), bf, "out")}, lambda o: ok(lib.tdb200_gate_residual(
        P(x16), P(y16), P(sc), P(o["out"]), BF, m, n, S())))
    cases["tdb200_gate_residual_stats"] = lambda: (
        {"out": ((m, n), bf, "out"), "row_stats": ((m, 2), f32, "out")},
        lambda o: ok(lib.tdb200_gate_residual_stats(P(x16), P(y16), P(sc), P(o["out"]), P(o["row_stats"]), BF, m, n, eps, S())))
    stats = torch.stack([x32.mean(1), torch.rsqrt(x32.var(1, unbiased=False) + eps)], 1).contiguous()
    cases["tdb200_layer_norm_modulate_quant_stats"] = lambda: (quant_specs, lambda o: ok(
        lib.tdb200_layer_norm_modulate_quant_stats(P(x16), BF, P(stats), P(sc), P(sh), P(o["q"]), P(o["s"]), m, n, S())))
    # a6 RoPE
    hd = 128
    heads = n // hd
    ang = torch.rand(m, hd // 2, device=dev, generator=g) * 20
    cos_sin = torch.stack([ang.cos(), ang.sin()], -1).contiguous()
    cases["tdb200_rope_interleaved"] = lambda: ({"y": ((m, n), bf, "out")}, lambda o: ok(lib.tdb200_rope_interleaved(
        P(x16), BF, P(ang), P(o["y"]), m, heads, hd, S())))
    cases["tdb200_rms_norm_rope"] = lambda: ({"y": ((m, n), bf, "out")}, lambda o: ok(lib.tdb200_rms_norm_rope(
        P(x16), BF, P(w), P(ang), P(o["y"]), m, heads, hd, eps, S())))
    cases["tdb200_rms_norm_rope_table"] = lambda: ({"y": ((m, n), bf, "out")}, lambda o: ok(lib.tdb200_rms_norm_rope_table(
        P(x16), BF, P(w), P(cos_sin), P(o["y"]), m, heads, hd, eps, S())))

    # a7-a10 SLA
    b, l, h, d = sz["sla"]
    q, v = rnd(b, l, h, d), rnd(b, l, h, d)
    kk = (torch.randn(b, l, h, d, device=dev, generator=g) + 2 * torch.randn(b, 1, h, d, device=dev, generator=g)).to(bf)
    mblk, nblk = cdiv(l, 128), cdiv(l, 64)
    topk = max(1, nblk // 10)
    cases["tdb200_sla_quant_qk"] = lambda: (
        {"kmean": ((b, h, d), f32, "out"), "q_i8": ((b, h, l, d), i8, "out"), "q_scale": ((b, h, mblk), f32, "out"),
         "k_i8": ((b, h, l, d), i8, "out"), "k_scale": ((b, h, nblk), f32, "out"), "q_pool": ((b, h, mblk, d), bf, "out"),
         "k_pool": ((b, h, nblk, d), bf, "out")},
        lambda o: ok(lib.tdb200_sla_quant_qk(P(q), P(kk), BF, b, l, l, h, d, P(o["kmean"]), P(o["q_i8"]), P(o["q_scale"]),
                                             P(o["k_i8"]), P(o["k_scale"]), P(o["q_pool"]), P(o["k_pool"]), S())))
    prep = quant_qk(q, kk)
    cases["tdb200_sla_block_map"] = lambda: (
        {"sparse_map": ((b, h, mblk, nblk), i8, "out"), "lut": ((b, h, mblk, topk), i32, "out")},
        lambda o: ok(lib.tdb200_sla_block_map(P(prep.q_pool), P(prep.k_pool), BF, b, h, mblk, nblk, d, topk,
                                              P(o["sparse_map"]), P(o["lut"]), S())))

    def moments_case(kx, vx):
        bx, lx, hx, dx = kx.shape
        nbytes = moments_workspace_bytes(bx, lx, hx, dx)
        pre = {"kv": rnd(bx, hx, dx, dx, dtype=f32), "ksum": rnd(bx, hx, dx, dtype=f32)}
        return ({"kv": ((bx, hx, dx, dx), f32, "acc"), "ksum": ((bx, hx, dx), f32, "acc"), "ws": ((nbytes,), torch.uint8, "ws")},
                lambda o: ok(lib.tdb200_sla_linear_moments_ws(P(kx), P(vx), BF, bx, lx, hx, dx, 0, P(o["kv"]), P(o["ksum"]),
                                                              P(o["ws"]), nbytes, S())),
                pre)
    cases["tdb200_sla_linear_moments_ws"] = lambda: moments_case(kk, v)
    # 64-wide heads run as pairs of heads; an odd head count leaves the last pair half empty
    k64, v64 = (t.reshape(b, l, 2 * h, 64)[:, :, : 2 * h - 1].contiguous() for t in (kk, v))
    cases["tdb200_sla_linear_moments_ws[d64,odd heads]"] = lambda: moments_case(k64, v64)
    kv, ksum = linear_moments(kk, v)
    proj_w, proj_b = rnd(d, d, scale=0.05, dtype=f32), rnd(d, scale=0.05, dtype=f32)
    cases["tdb200_sla_project_moments"] = lambda: ({"kvw": ((b, h, d, d), bf, "out")}, lambda o: ok(
        lib.tdb200_sla_project_moments(P(proj_w), P(kv), BF, b * h, d, P(o["kvw"]), S())))
    kvw = project_moments(proj_w, kv, bf)
    _, lut = block_map_from_pools(prep.q_pool, prep.k_pool, topk)
    sm = d ** -0.5
    out_spec = {"out": ((b, l, h, d), bf, "out")}
    cases["tdb200_sla_attn_fwd"] = lambda: (out_spec, lambda o: ok(lib.tdb200_sla_attn_fwd(
        P(prep.q_i8), P(prep.q_scale), P(prep.k_i8), P(prep.k_scale), P(v), P(q), BF, P(lut), topk, P(kvw), P(ksum),
        P(proj_b), P(o["out"]), b, l, l, h, d, sm, S())))
    cases["tdb200_sla_attn_fwd_v2"] = lambda: (out_spec, lambda o: ok(lib.tdb200_sla_attn_fwd_v2(
        P(prep.q_i8), P(prep.q_scale), P(prep.k_i8), P(prep.k_scale), P(v), P(q), BF, P(lut), topk, P(kvw), P(ksum),
        P(proj_b), P(o["out"]), b, l, l, h, d, sm, 0, S())))
    cases["tdb200_sla_attn_fwd_qk16"] = lambda: (out_spec, lambda o: ok(lib.tdb200_sla_attn_fwd_qk16(
        P(q), P(kk), P(v), BF, P(lut), topk, P(kvw), P(ksum), P(proj_b), P(o["out"]), b, l, l, h, d, sm, S())))
    chunks = cdiv(l, 128)
    cases["tdb200_sla_kmean_partial"] = lambda: ({"partial": ((b, h, chunks, d), f32, "out")}, lambda o: ok(
        lib.tdb200_sla_kmean_partial(P(kk), BF, b, l, h, d, P(o["partial"]), S())))
    partial = torch.randn(b, h, chunks, d, device=dev, generator=g) * l / 10
    cases["tdb200_sla_kmean_final"] = lambda: ({"kmean": ((b, h, d), f32, "out")}, lambda o: ok(
        lib.tdb200_sla_kmean_final(P(partial), b, h, chunks, d, l, P(o["kmean"]), S())))
    k1, v1, q1 = kk[:1].contiguous(), v[:1].contiguous(), q[:1].contiguous()   # the sequence-major K layout is one sequence
    prep1 = quant_qk(q1, k1)
    cases["tdb200_sla_quant_k_seq"] = lambda: (
        {"k_i8": ((1, l, h, d), i8, "out"), "k_scale": ((1, h, nblk), f32, "out"), "k_pool": ((1, h, nblk, d), bf, "out")},
        lambda o: ok(lib.tdb200_sla_quant_k_seq(P(k1), P(prep1.kmean), BF, 1, l, h, d, P(o["k_i8"]), P(o["k_scale"]),
                                                P(o["k_pool"]), S())))
    ks_i8, ks_scale, _ = quant_k_seq(k1, prep1.kmean)
    lut1 = lut[:1].contiguous()
    cases["tdb200_sla_attn_fwd_kseq"] = lambda: ({"out": ((1, l, h, d), bf, "out")}, lambda o: ok(
        lib.tdb200_sla_attn_fwd_kseq(P(prep1.q_i8), P(prep1.q_scale), P(ks_i8), P(ks_scale), P(v1), P(q1), BF, P(lut1), topk,
                                     P(kvw), P(ksum), P(proj_b), P(o["out"]), 1, l, l, h, d, sm, S())))

    # a12 LTX-2
    lb, lt, ln = sz["ltx"]
    xl, rl = rnd(lb, lt, ln), rnd(lb, lt, ln)
    table = rnd(6, ln, scale=0.1, dtype=f32)
    ts = rnd(lb, 1, 6 * ln, scale=0.1)
    yl = {"y": ((lb, lt, ln), bf, "out")}
    cases["tdb200_ltx_modulated_rms_norm_ada"] = lambda: (yl, lambda o: ok(lib.tdb200_ltx_modulated_rms_norm_ada(
        P(xl), BF, P(table), P(ts), 1, 0, 6, P(o["y"]), lb, lt, 1, ln, eps, S())))
    cases["tdb200_ltx_modulate_ada"] = lambda: (yl, lambda o: ok(lib.tdb200_ltx_modulate_ada(
        P(xl), BF, P(table), P(ts), 4, 3, 6, P(o["y"]), lb, lt, 1, ln, S())))
    cases["tdb200_ltx_gated_residual_ada"] = lambda: (yl, lambda o: ok(lib.tdb200_ltx_gated_residual_ada(
        P(xl), P(rl), BF, P(table), P(ts), 2, 6, P(o["y"]), lb, lt, 1, ln, S())))
    lh, ld = ln // 128, 128
    cosf, sinf = rnd(lb, lh, lt, ld // 2), rnd(lb, lh, lt, ld // 2)
    cases["tdb200_ltx_split_rope"] = lambda: (yl, lambda o: ok(lib.tdb200_ltx_split_rope(
        P(xl), P(cosf), P(sinf), BF, P(o["y"]), lb, lt, lh, ld, S())))
    cases["tdb200_quant_int8_rowwise"] = lambda: ({"q": ((m, n), i8, "out"), "s": ((m,), f32, "out")}, lambda o: ok(
        lib.tdb200_quant_int8_rowwise(P(x16), BF, m, n, P(o["q"]), P(o["s"]), S())))
    ra_s, rb_s = torch.rand(m, device=dev, generator=g) * 0.01, torch.rand(ffn, device=dev, generator=g) * 0.01
    cases["tdb200_gemm_w8a8_rowwise"] = lambda: ({"c": ((m, ffn), bf, "out")}, lambda o: ok(lib.tdb200_gemm_w8a8_rowwise(
        P(a_q), P(ra_s), P(b_q), P(rb_s), P(bias), P(o["c"]), BF, m, ffn, k, S())))
    return cases


# Entry points deliberately outside the rerun check: the moments entry points without a workspace add their split partials
# with fp32 atomics (documented as run-order dependent), and the diagnostics.
NOT_RERUN = {"tdb200_abi_version", "tdb200_last_error", "tdb200_sla_linear_moments", "tdb200_sla_linear_moments_ex",
             "tdb200_sla_linear_moments_workspace", "tdb200_debug_set_attn_trace", "tdb200_selftest_umma_bf16",
             "tdb200_selftest_tmem_read", "tdb200_selftest_mufu", "tdb200_selftest_softmax_exps"}


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["small", "A"])
def test_every_entry_point_reruns_bit_identically_and_writes_every_output(cuda, size):
    from turbodiffusion_b200 import _lib
    cases = _cases(SIZES[size], cuda)
    covered = {name.split("[")[0] for name in cases}
    assert covered == set(_lib.exported_names()) - NOT_RERUN, "an entry point of tdb200.h has no rerun case"
    failures = []
    for name, build in cases.items():
        specs, call, *pre = build()
        prefill = pre[0] if pre else None
        try:
            got = check_rerun_with_poison(specs, call, cuda, prefill)
            if prefill:   # accumulators: prefill + (the zero-prefill result), with one fp32 rounding
                zero = check_rerun_with_poison(specs, call, cuda, {n: torch.zeros_like(t) for n, t in prefill.items()})
                for acc, t in prefill.items():
                    assert torch.equal(got[acc], t + zero[acc]), f"{acc}: result != prefill + zero-prefill result"
        except AssertionError as ex:
            failures.append(f"{name}: {ex}")
    assert not failures, "\n".join(failures)


@pytest.mark.gpu
@pytest.mark.parametrize("b,l,h,d", [(1, 32760, 12, 128), (2, 1305, 3, 128), (1, 1305, 5, 64), (3, 200, 40, 128)])
def test_reproducible_moments_equal_the_atomic_ones(cuda, b, l, h, d):
    """The fixed-order reduction computes the sums the atomic entry point computes, up to fp32 summation order."""
    from turbodiffusion_b200._lib import DTYPE_TAG, lib, ptr, stream_ptr
    from turbodiffusion_b200.SLA.core import linear_moments
    g = torch.Generator(device=cuda).manual_seed(3)
    k = torch.randn(b, l, h, d, device=cuda, generator=g).bfloat16()
    v = torch.randn(b, l, h, d, device=cuda, generator=g).bfloat16()
    kv, ksum = linear_moments(k, v)
    kv_a, ksum_a = torch.zeros_like(kv), torch.zeros_like(ksum)
    assert lib().tdb200_sla_linear_moments_ex(ptr(k), ptr(v), DTYPE_TAG[k.dtype], b, l, h, d, 0, ptr(kv_a), ptr(ksum_a),
                                              stream_ptr(k.device)) == 0
    for got, ref in ((kv, kv_a), (ksum, ksum_a)):
        st = O.stats(got.cpu(), ref.cpu())
        assert st["rel_l2"] < 1e-6, st
    assert torch.allclose(ksum.sum(-1), torch.full_like(ksum[..., 0], float(l)), rtol=1e-3)   # softmax rows sum to one
    kv2, ksum2 = linear_moments(k, v)
    assert torch.equal(kv, kv2) and torch.equal(ksum, ksum2)


# ---- (b) the denoise step at the real width -------------------------------------------------------------------------------
# Wan-1.3B: dim 1536, 12 heads of 128, FFN 8960, 512 text tokens.  thw (3, 15, 29): L = 1305, ragged query (25 of 128 rows)
# and key (25 of 64 rows) tails; (21, 30, 52): shape A, L = 32760.
STEP_CASES = [((3, 15, 29), 3), ((21, 30, 52), 2)]


def _hot_path(cuda, thw, layers, attention="sagesla"):
    from turbodiffusion_b200.block import WanBlockB200, WanHotPath, random_block_state
    from turbodiffusion_b200.ops import wan_rope_angles
    dim, ffn, heads, text = 1536, 8960, 12, 512
    model = WanHotPath(dim, ffn, heads, layers, cuda, seed=1234)
    if attention != "sagesla":
        model.blocks = [WanBlockB200(random_block_state(dim, ffn, heads, 1234 + i, cuda), dim, heads, topk=0.1,
                                     attention=attention) for i in range(layers)]
    l = thw[0] * thw[1] * thw[2]
    g = torch.Generator().manual_seed(7)
    x = torch.randn(l, dim, generator=g).bfloat16().to(cuda)
    e0 = (torch.randn(6, dim, generator=g) * 0.1).to(cuda)
    ctx = torch.randn(text, dim, generator=g).bfloat16().to(cuda)
    ang = wan_rope_angles(*thw, dim // heads).to(cuda)
    return model, x, e0, ang, ctx


def _chained(model, x, e0, ang, ctx, keep=None):
    """The step's blocks one after the other, each forming its own LayerNorm statistics and modulation table."""
    for blk in model.blocks:
        if keep is not None:
            blk.sla._keep_selection = {}
        x_in = x
        x = blk(x, e0, ang, ctx)
        if keep is not None:
            keep.append((x_in, x, blk.sla._keep_selection["lut"]))
            blk.sla._keep_selection = None
    return x


def _bits_equal(a, b, what):
    neq = a.view(torch.int16) != b.view(torch.int16)
    assert not neq.any(), (f"{what}: {neq.sum().item()} of {neq.numel()} elements differ; max abs "
                           f"{(a.float() - b.float()).abs().max().item():.4g}; first {neq.nonzero()[:3].tolist()}")


@pytest.mark.gpu
@pytest.mark.parametrize("thw,layers", STEP_CASES)
def test_step_is_bit_reproducible_in_eager_graph_and_unfused_form(cuda, thw, layers):
    model, x, e0, ang, ctx = _hot_path(cuda, thw, layers)
    y1 = model.step(x, e0, ang, ctx)
    y2 = model.step(x, e0, ang, ctx)
    _bits_equal(y1, y2, "two eager steps")

    # captured like bench.run_b200: one warm-up step on a side stream, capture, replay
    xs, es, cs = x.clone(), e0.clone(), ctx.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        model.step(xs, es, ang, cs)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ys = model.step(xs, es, ang, cs)
    graph.replay()
    torch.cuda.synchronize()
    _bits_equal(ys, y1, "graph replay vs eager step")
    graph.replay()
    torch.cuda.synchronize()
    _bits_equal(ys, y1, "second graph replay vs eager step")
    del graph

    _bits_equal(_chained(model, x, e0, ang, ctx), y1, "step() vs blocks chained with stats=None, e=None")


# ---- (c) every layer against the CPU oracle ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("attention", ["sagesla", "sla"])
def test_every_layer_of_the_step_matches_the_oracle(cuda, attention):
    """Each layer's GPU output against oracle.wan_block_forward on that layer's GPU input and the kernel's own block selection:
    the oracle's drift cannot add up across layers, while a fault of one layer or of the chaining still shows."""
    thw, layers = STEP_CASES[0]
    model, x, e0, ang, ctx = _hot_path(cuda, thw, layers, attention)
    keep = []
    y = _chained(model, x, e0, ang, ctx, keep)
    _bits_equal(model.step(x, e0, ang, ctx), y, "step() vs chained blocks")
    e0c, angc, ctxc = e0.cpu(), ang.cpu(), ctx.cpu()
    for i, (blk, (x_in, x_out, lut)) in enumerate(zip(model.blocks, keep)):
        sd = {k: v.cpu() for k, v in blk.sd.items()}
        ref = O.wan_block_forward(sd, x_in.cpu(), e0c, angc, ctxc, blk.dim, blk.heads, lut=lut.cpu())
        st = O.stats(x_out.cpu(), ref)
        assert st["cos"] > 0.9995 and st["rel_l2"] < 2.5e-2, (i, st)


# ---- (d) W8A8 GEMM at the real K and N -------------------------------------------------------------------------------------
def _sampled_rows(m):
    """One interior 128-row tile and the ragged last tile: whole tiles, so the oracle's per-128-row scales line up."""
    mid = (m // 128) // 2
    last = (m - 1) // 128
    rows = torch.cat([torch.arange(mid * 128, mid * 128 + 128), torch.arange(last * 128, m)])
    return rows, torch.tensor([mid, last])


def _gemm_operands(cuda, m, n, k, seed):
    g = torch.Generator(device=cuda).manual_seed(seed)
    a_q = torch.randint(-128, 128, (m, k), device=cuda, generator=g, dtype=torch.int8)
    b_q = torch.randint(-128, 128, (n, k), device=cuda, generator=g, dtype=torch.int8)
    a_s = torch.rand((m + 127) // 128, k // 128, device=cuda, generator=g) * 1e-3 + 1e-5
    b_s = torch.rand((n + 127) // 128, k // 128, device=cuda, generator=g) * 1e-3 + 1e-5
    return a_q, a_s, b_q, b_s


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,k", [(32760, 8960, 1536), (32760, 1536, 8960), (75600, 13824, 5120), (75600, 5120, 13824)])
def test_gemm_bit_exact_at_real_k_and_n(cuda, m, n, k):
    from turbodiffusion_b200.turbo_diffusion_ops import gemm_cuda
    a_q, a_s, b_q, b_s = _gemm_operands(cuda, m, n, k, seed=m + n + k)
    c = torch.full((m, n), float("nan"), dtype=torch.bfloat16, device=cuda)
    gemm_cuda(a_q, a_s, b_q, b_s, c)
    torch.cuda.synchronize()
    assert not torch.isnan(c).any().item(), "some outputs were never written"
    rows, tiles = _sampled_rows(m)
    ref = O.int8_gemm(a_q[rows.to(cuda)].cpu(), a_s[tiles.to(cuda)].cpu(), b_q.cpu(), b_s.cpu(), torch.bfloat16)
    _bits_equal(c[rows.to(cuda)].cpu(), ref, f"rows {rows[0].item()}.. and the ragged tail of {m}x{n}x{k}")


@pytest.mark.gpu
def test_gemm_quant_out_bit_exact_at_the_ffn_up_shape(cuda):
    from turbodiffusion_b200.turbo_diffusion_ops import gemm_cuda_quant_out
    m, n, k = 32760, 8960, 1536
    a_q, a_s, b_q, b_s = _gemm_operands(cuda, m, n, k, seed=5)
    q, s = gemm_cuda_quant_out(a_q, a_s, b_q, b_s, None, torch.bfloat16, gelu=False)
    torch.cuda.synchronize()
    rows, tiles = _sampled_rows(m)
    mid = O.int8_gemm(a_q[rows.to(cuda)].cpu(), a_s[tiles.to(cuda)].cpu(), b_q.cpu(), b_s.cpu(), torch.bfloat16)
    q_ref, s_ref = O.int8_quant(mid)
    assert torch.equal(s[tiles.to(cuda)].cpu(), s_ref), "block scales differ"
    neq = q[rows.to(cuda)].cpu() != q_ref
    assert not neq.any(), f"{neq.sum().item()} int8 codes differ; first {neq.nonzero()[:3].tolist()}"
