"""CPU restatement of TurboDiffusion's denoise hot path — TEST INFRASTRUCTURE ONLY.

This module is the *oracle*: a plain torch-on-CPU (plus a small C helper, oracle/td_oracle_c.c) restatement of the
reference algorithm with the reference's exact rounding points.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import it.  The product (turbodiffusion_b200) never does.

Every function cites the reference file:line it follows (paths relative to thu-ml/TurboDiffusion).

Pinning status (see tests/test_oracle_vs_reference.py and tests/golden/):
  * norms, mean_pool, get_block_map, sparse attention (_attn_fwd), SparseLinearAttention.forward:
      pinned against the reference's OWN Triton kernels / torch code executed on CPU with TRITON_INTERPRET=1
      (tools/make_golden.py imports /root/reference and writes tests/golden/*.pt).
  * LTX modulation helpers: pinned against the reference's known-answer tests
      (TurboT2AV/LTX-2/packages/ltx-core/tests/test_transformer_fusion_helpers.py:13-87).
  * int8_quant / int8 GEMM: the reference implementation is CUDA-only (ops/quant/quant.hpp, ops/gemm/kernel.hpp);
      restated from the source; cross-checked on the GPU against the reference extension when oracle/_ref holds a
      build of it.  Golden vectors are generated from this restatement.
  * Sage INT8 quantisation + attention arithmetic (third-party thu-ml/SpargeAttn @ ae5b629e, not in the tree):
      PARITY UNPINNED.  `sage_*` functions restate the published algorithm (SageAttention2 / SpargeAttn README and
      the call sites SLA/core.py:197-235) and are labelled as an emulation.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional, Tuple

import torch
import torch.nn.functional as F

_HERE = os.path.dirname(os.path.abspath(__file__))
_C = None


def _c_lib():
    """oracle/libtd_oracle_c.so (built by __graft_entry__.build()); None if absent."""
    global _C
    if _C is None:
        path = os.path.join(_HERE, "libtd_oracle_c.so")
        if os.path.exists(path):
            lib = ctypes.CDLL(path)
            lib.td_w8a8_gemm_f32.restype = None
            lib.td_w8a8_gemm_f32.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int64] * 3
            _C = lib
        else:
            _C = False
    return _C or None


def next_pow2(n: int) -> int:
    return 1 << (int(n) - 1).bit_length()


def cdiv(a: int, b: int) -> int:
    return (a + b - 1) // b


# =============================================================================================
# a1. int8_quant  — ops/quant/quant.hpp:86-99 (scale), :122-154 (amax), :157-163 (convert), common/store.hpp:46
# =============================================================================================
def int8_quant(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """x [M,K] bf16/fp16 -> (q int8 [M,K], s fp32 [ceil(M/128), ceil(K/128)]).

    Per 128x128 block (ragged edges: only in-range elements, load.hpp:33-36 loads 0 elsewhere):
      amax = max(1e-8, max|x|);  s = amax/128;  q = sat_s8(rint(x * (128/amax)))   (cvt.rni.sat.s8.f32)
    The device computes 128/amax with div.approx under --use_fast_math (setup.py:34); this restatement uses the IEEE
    quotient, so reference-device codes may differ by one at exact .5 ties; scales are bit-identical.
    """
    assert x.dim() == 2 and x.dtype in (torch.bfloat16, torch.float16)
    m, k = x.shape
    mb, kb = cdiv(m, 128), cdiv(k, 128)
    xf = torch.zeros(mb * 128, kb * 128, dtype=torch.float32)
    xf[:m, :k] = x.float()
    blocks = xf.view(mb, 128, kb, 128)
    amax = blocks.abs().amax(dim=(1, 3)).clamp_min(1e-8)  # [mb, kb]
    s = amax / 128.0
    r = (torch.tensor(128.0) / amax).to(torch.float32)
    y = blocks * r[:, None, :, None]
    q = torch.round(y).clamp_(-128, 127).to(torch.int8)  # torch.round = half-to-even = rni
    return q.view(mb * 128, kb * 128)[:m, :k].contiguous(), s.contiguous()


# =============================================================================================
# a2. W8A8 GEMM — ops/gemm/kernel.hpp:391-427 (per-K-block order), utils.hpp:116-121 (fma with the scale product),
#     output cast kernel.hpp:471-477; bias add ops/core.py:410-411
# =============================================================================================
def int8_gemm_f32(a_q: torch.Tensor, a_s: torch.Tensor, b_q: torch.Tensor, b_s: torch.Tensor) -> torch.Tensor:
    """fp32 accumulator before the output cast:  acc = fma(float(int_dot_kb), a_s[mb,kb]*b_s[nb,kb], acc), kb ascending."""
    m, k = a_q.shape
    n = b_q.shape[0]
    assert b_q.shape[1] == k and k % 128 == 0
    lib = _c_lib()
    a_q, b_q = a_q.contiguous(), b_q.contiguous()
    a_s, b_s = a_s.contiguous().float(), b_s.contiguous().float()
    if lib is not None:
        out = torch.empty(m, n, dtype=torch.float32)
        lib.td_w8a8_gemm_f32(a_q.data_ptr(), a_s.data_ptr(), b_q.data_ptr(), b_s.data_ptr(), out.data_ptr(), m, n, k)
        return out
    return _int8_gemm_f32_torch(a_q, a_s, b_q, b_s)


def _int8_gemm_f32_torch(a_q, a_s, b_q, b_s) -> torch.Tensor:
    """Pure-torch version: the product int*scale is exact in fp64 (22 + 24 bits); the fp64 sum rounded to fp32
    equals the fused fp32 FMA except for double-rounding ties (probability ~2^-29 per term)."""
    m, k = a_q.shape
    n = b_q.shape[0]
    acc = torch.zeros(m, n, dtype=torch.float32)
    rows = torch.arange(m) // 128
    cols = torch.arange(n) // 128
    for kb in range(k // 128):
        a = a_q[:, kb * 128:(kb + 1) * 128].float()
        b = b_q[:, kb * 128:(kb + 1) * 128].float()
        dot = a @ b.t()  # exact: integers, |sum| <= 128*128*128 < 2^24
        scale = (a_s[rows, kb][:, None] * b_s[cols, kb][None, :])  # fp32 product formed first
        acc = (dot.double() * scale.double() + acc.double()).float()
    return acc


def int8_gemm(a_q, a_s, b_q, b_s, out_dtype=torch.bfloat16, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    y = int8_gemm_f32(a_q, a_s, b_q, b_s).to(out_dtype)
    if bias is not None:
        y = y + bias.to(out_dtype)  # separate elementwise op in the module (ops/core.py:410-411)
    return y


def int8_linear(x: torch.Tensor, w_q: torch.Tensor, w_s: torch.Tensor, bias: Optional[torch.Tensor] = None):
    """ops/core.py:28-57 + Int8Linear.forward :408-412."""
    shape = x.shape
    x2 = x.reshape(-1, shape[-1])
    a_q, a_s = int8_quant(x2)
    y = int8_gemm(a_q, a_s, w_q, w_s, x.dtype, bias)
    return y.reshape(*shape[:-1], w_q.shape[0])


# =============================================================================================
# a3/a4. FastNorm — Triton kernels ops/core.py:96-136 (RMS), :193-243 / :293-335 (LayerNorm)
# =============================================================================================
def rmsnorm_f32(x: torch.Tensor, w: torch.Tensor, eps: float) -> torch.Tensor:
    """ops/core.py:121-135: var = sum(x^2)/N, rstd = 1/sqrt(var+eps), y = x*rstd*w (fp32)."""
    x = x.float()
    var = (x * x).sum(-1, keepdim=True) / x.shape[-1]
    rstd = 1.0 / torch.sqrt(var + eps)
    return (x * rstd) * w.float()


def layernorm_f32(x: torch.Tensor, w: Optional[torch.Tensor], b: Optional[torch.Tensor], eps: float,
                  reference_padding_quirk: bool = True) -> torch.Tensor:
    """ops/core.py:219-240 / :317-333.  NOTE the reference quirk: columns are padded to N2 = next_pow2(N) with 0
    (`tl.load(..., other=0.0)`, :217/:315) and the variance term `(x - mean)^2` is NOT masked (:222/:320), so every
    padded column contributes mean^2:   var = (sum_{j<N}(x_j-mean)^2 + (N2-N)*mean^2) / N.
    reference_padding_quirk=False gives the textbook biased variance instead."""
    x = x.float()
    n = x.shape[-1]
    mean = x.sum(-1, keepdim=True) / n
    d = x - mean
    ssq = (d * d).sum(-1, keepdim=True)
    if reference_padding_quirk:
        ssq = ssq + float(next_pow2(n) - n) * (mean * mean)
    var = ssq / n
    rstd = 1.0 / torch.sqrt(var + eps)
    y = d * rstd
    if w is not None:
        y = y * w.float() + (b.float() if b is not None else 0.0)
    return y


def fast_rmsnorm(x: torch.Tensor, w: torch.Tensor, eps: float) -> torch.Tensor:
    """FastRMSNorm.forward, ops/core.py:441-442: rmsnorm(x.float(), w, eps).to(x.dtype)."""
    return rmsnorm_f32(x, w, eps).to(x.dtype)


def fast_layernorm(x, w, b, eps) -> torch.Tensor:
    """FastLayerNorm.forward, ops/core.py:477-478."""
    return layernorm_f32(x, w, b, eps).to(x.dtype)


# =============================================================================================
# a5. AdaLN modulation / gate — rcm/networks/wan2pt1.py:398-417
# =============================================================================================
def ln_modulate(x: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, eps: float) -> torch.Tensor:
    """wan2pt1.py:403-404: (norm1(x).float() * (1 + e[1]) + e[0]).type_as(x); norm1 = FastLayerNorm (no affine).
    The LayerNorm result is rounded to x.dtype before the modulation."""
    h = fast_layernorm(x, None, None, eps)
    return (h.float() * (1.0 + scale.float()) + shift.float()).to(x.dtype)


def gate_residual(x: torch.Tensor, y: torch.Tensor, gate: torch.Tensor) -> torch.Tensor:
    """wan2pt1.py:405-406 (`x = x + y * e[2].type_as(x)` with bf16 tensors under an fp32 autocast context, which does
    not touch elementwise ops): out = T(x + T(y * T(gate)))."""
    g = gate.to(x.dtype)
    return x + y * g


# =============================================================================================
# a6. RoPE — rcm/networks/wan2pt1.py:156-178 (flash_attn apply_rotary_emb, interleaved=True)
# =============================================================================================
def rope_interleaved(x: torch.Tensor, angles: torch.Tensor) -> torch.Tensor:
    """x [..., L, H, D], angles [L, D/2] fp32.  Pairs (2i, 2i+1): o0 = x0*c - x1*s, o1 = x0*s + x1*c in fp32."""
    xf = x.float()
    c = torch.cos(angles.float())[:, None, :]
    s = torch.sin(angles.float())[:, None, :]
    x0, x1 = xf[..., 0::2], xf[..., 1::2]
    o = torch.empty_like(xf)
    o[..., 0::2] = x0 * c - x1 * s
    o[..., 1::2] = x0 * s + x1 * c
    return o.to(x.dtype)


def rms_norm_rope(x: torch.Tensor, w: torch.Tensor, angles: torch.Tensor, eps: float) -> torch.Tensor:
    """WanSelfAttention.forward, wan2pt1.py:261-268: norm_q over the FULL model dim, view as heads, rope_apply."""
    l, h, d = x.shape[-3:]
    y = fast_rmsnorm(x.reshape(*x.shape[:-2], h * d), w, eps).reshape(x.shape)
    return rope_interleaved(y, angles)


def wan_rope_angles(t: int, hh: int, ww: int, d: int) -> torch.Tensor:
    """VideoRopePosition3DEmb.generate_embeddings, wan2pt1.py:111-137 with the Wan split d_h = d_w = 2*(d//6),
    d_t = d - 2*d_h; theta = 10000, ntk factors 1.  Returns [t*hh*ww, d/2] fp32 angles."""
    dh = dw = d // 6 * 2
    dt = d - 2 * dh

    def freqs(dim):
        rng = torch.arange(0, dim, 2)[: dim // 2].float() / dim
        return 1.0 / (10000.0 ** rng)

    seq = torch.arange(max(t, hh, ww)).float()
    ft = torch.outer(seq[:t], freqs(dt))
    fh = torch.outer(seq[:hh], freqs(dh))
    fw = torch.outer(seq[:ww], freqs(dw))
    out = torch.cat([ft[:, None, None, :].expand(t, hh, ww, -1), fh[None, :, None, :].expand(t, hh, ww, -1),
                     fw[None, None, :, :].expand(t, hh, ww, -1)], dim=-1)
    return out.reshape(t * hh * ww, d // 2).float().contiguous()


# =============================================================================================
# a7. block map — SLA/utils.py:21-52 (mean_pool), :55-67 (get_block_map)
# =============================================================================================
def mean_pool(x: torch.Tensor, blk: int) -> torch.Tensor:
    """x [B,H,L,D] -> [B,H,ceil(L/blk),D] in x.dtype; fp32 sum divided by the ACTUAL row count of the block (:38-40)."""
    b, h, l, d = x.shape
    nb = cdiv(l, blk)
    pad = nb * blk - l
    xf = x.float()
    if pad:
        xf = F.pad(xf, (0, 0, 0, pad))
    sums = xf.view(b, h, nb, blk, d).sum(3)
    cnt = torch.full((nb,), float(blk))
    cnt[-1] = float(l - (nb - 1) * blk)
    return (sums / cnt[None, None, :, None]).to(x.dtype)


def smooth_k(k: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """SLA/utils.py:56: arg_k = k - mean_L(k) evaluated in k.dtype.  Returns (arg_k, km) both in k.dtype."""
    km = torch.mean(k, dim=-2, keepdim=True)
    return k - km, km


def pooled_scores(q: torch.Tensor, k: torch.Tensor, blkq: int, blkk: int) -> torch.Tensor:
    """SLA/utils.py:56-59: T(Qpool . Kpool^T) with Kpool pooled from the smoothed keys.  q,k [B,H,L,D]."""
    arg_k, _ = smooth_k(k)
    pq = mean_pool(q, blkq)
    pk = mean_pool(arg_k, blkk)
    return (pq.float() @ pk.float().transpose(-1, -2)).to(q.dtype)


def select_topk(scores: torch.Tensor, topk: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Top-`topk` block ids per row with the tie rule 'lowest index first' (torch.topk(sorted=False) leaves ties
    implementation-defined; SageSLA only consumes the SET, SLA/core.py:204).  Returns (sparse_map int8, lut int32
    ascending)."""
    s = scores.float()
    order = torch.argsort(s, dim=-1, descending=True, stable=True)  # stable -> lowest index first among equals
    sel = order[..., :topk]
    sparse_map = torch.zeros(scores.shape, dtype=torch.int8)
    sparse_map.scatter_(-1, sel, 1)
    lut = torch.sort(sel, dim=-1).values.to(torch.int32)
    return sparse_map, lut


def get_block_map(q: torch.Tensor, k: torch.Tensor, topk_ratio: float, blkq: int = 128, blkk: int = 64):
    """SLA/utils.py:55-67.  q,k [B,H,L,D].  Returns (sparse_map int8 [B,H,Mblk,Nblk], lut int32 ascending, topk)."""
    scores = pooled_scores(q, k, blkq, blkk)
    nblk = scores.shape[-1]
    topk = min(nblk, int(topk_ratio * nblk))
    sparse_map, lut = select_topk(scores, topk)
    return sparse_map, lut, topk


# =============================================================================================
# a8. Sage Q/K quantisation — third party (SpargeAttn get_vanilla_qk_quant), call site SLA/core.py:200-203.
#     EMULATION, parity unpinned.
# =============================================================================================
def sage_quant_blocks(x: torch.Tensor, blk: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """x [B,H,L,D] (bf16/fp16) -> (int8 [B,H,L,D], scale fp32 [B,H,ceil(L/blk)]).
    Per block of `blk` rows: scale = max|x|/127 + 1e-7;  q = trunc(x/scale + 0.5*sign(x))  (round half away)."""
    b, h, l, d = x.shape
    nb = cdiv(l, blk)
    xf = x.float()
    pad = nb * blk - l
    if pad:
        xf = F.pad(xf, (0, 0, 0, pad))
    blocks = xf.view(b, h, nb, blk, d)
    scale = blocks.abs().amax(dim=(3, 4)) / 127.0 + 1e-7
    y = blocks / scale[..., None, None]
    y = y + 0.5 * torch.where(y >= 0, 1.0, -1.0)
    qi = y.to(torch.int32).clamp_(-128, 127).to(torch.int8)  # .to(int) truncates toward zero like tl's .to(int8)
    return qi.view(b, h, nb * blk, d)[:, :, :l].contiguous(), scale.contiguous()


def sage_quant_qk(q: torch.Tensor, k: torch.Tensor, blkq: int = 128, blkk: int = 64):
    """q,k [B,H,L,D] in the compute dtype.  Returns q_i8, q_scale, k_i8 (of T(k - T(mean_L k))), k_scale, km."""
    arg_k, km = smooth_k(k)
    q_i8, q_s = sage_quant_blocks(q, blkq)
    k_i8, k_s = sage_quant_blocks(arg_k, blkk)
    return q_i8, q_s, k_i8, k_s, km


# =============================================================================================
# a9 / a9'. block-sparse softmax attention — SLA/kernel.py:33-82
# =============================================================================================
def sparse_attention(q, k, v, lut, blkq: int = 128, blkk: int = 64, sm_scale: Optional[float] = None,
                     p_dtype: Optional[torch.dtype] = None, q_i8=None, q_s=None, k_i8=None, k_s=None) -> torch.Tensor:
    """q,k,v [B,H,L,D]; lut [B,H,Mblk,topk] block ids.  Exact (fp32) softmax over the selected key blocks, columns
    >= L masked (SLA/kernel.py:57-62).  Returns fp32 [B,H,L,D].
      p_dtype=None            : the exact block-sparse oracle (no rounding of P)
      p_dtype=torch.bfloat16  : P rounded before P.V as the Triton kernel does (:73), row sum from unrounded P (:71)
      q_i8.. given            : scores from the INT8 emulation  (qi . ki) * q_s * k_s * sm_scale   [Sage, unpinned]
    """
    b, h, l, d = q.shape
    lk = k.shape[2]
    if sm_scale is None:
        sm_scale = d ** -0.5
    mblk = cdiv(l, blkq)
    out = torch.zeros(b, h, l, d, dtype=torch.float32)
    vf = v.float()
    use_i8 = q_i8 is not None
    kf = k_i8.float() if use_i8 else k.float()
    qf = q_i8.float() if use_i8 else q.float()
    for bi in range(b):
        for hi in range(h):
            for mi in range(mblk):
                r0, r1 = mi * blkq, min(l, (mi + 1) * blkq)
                ids = lut[bi, hi, mi].long()
                cols = (ids[:, None] * blkk + torch.arange(blkk)[None, :])  # [topk, blkk]
                valid = cols < lk
                cidx = cols.clamp_max(lk - 1).reshape(-1)
                s = qf[bi, hi, r0:r1] @ kf[bi, hi, cidx].t()
                if use_i8:
                    ks = k_s[bi, hi, ids][:, None].expand(-1, blkk).reshape(-1)
                    s = s * (q_s[bi, hi, mi] * sm_scale) * ks[None, :]
                else:
                    s = s * sm_scale
                s = s.masked_fill(~valid.reshape(-1)[None, :], float("-inf"))
                mrow = s.amax(-1, keepdim=True)
                p = torch.exp(s - mrow)
                lsum = p.sum(-1, keepdim=True)
                if p_dtype is not None:
                    p = p.to(p_dtype).float()
                out[bi, hi, r0:r1] = (p @ vf[bi, hi, cidx]) / lsum
    return out


def dense_attention(q, k, v, sm_scale: Optional[float] = None) -> torch.Tensor:
    """The reference's 'original' attention = F.scaled_dot_product_attention (rcm/utils/attention.py:152-166 body;
    the wrapper refuses CPU, see BASELINE.md §3).  q,k,v [B,H,L,D]."""
    return F.scaled_dot_product_attention(q, k, v, scale=sm_scale)


# =============================================================================================
# a10. linear branch + merge — SLA/core.py:243-253 (== :104-114)
# =============================================================================================
def linear_branch(q, k, v, proj_w: torch.Tensor, proj_b: torch.Tensor, dtype=torch.bfloat16,
                  exact: bool = False) -> torch.Tensor:
    """q,k,v [B,H,L,D] in `dtype`.  exact=False follows the reference's rounding points on CPU tensors of `dtype`
    (softmax -> dtype, kv bmm -> dtype, ...); exact=True keeps everything in fp32 (the better-than-reference target a
    fused kernel is judged against, SURVEY appendix A.8).  Returns o_l after proj_l, [B,H,L,D] (dtype or fp32)."""
    if exact:
        pq = torch.softmax(q.float(), -1).to(dtype).float()
        pk = torch.softmax(k.float(), -1).to(dtype).float()
        kv = pk.transpose(-1, -2) @ v.float()
        ks = pk.sum(-2, keepdim=True)
        o = (pq @ kv) / (1e-5 + (pq * ks).sum(-1, keepdim=True))
        return o @ proj_w.float().t() + proj_b.float()
    pq = torch.softmax(q, -1).contiguous().to(dtype)
    pk = torch.softmax(k, -1).contiguous().to(dtype)
    kvsum = pk.transpose(-1, -2) @ v
    ksum = torch.sum(pk, dim=-2, keepdim=True)
    o_l = (pq @ kvsum) / (1e-5 + (pq * ksum).sum(dim=-1, keepdim=True))
    # `with torch.amp.autocast('cuda', dtype)`: fp32 Linear evaluated in `dtype`
    return F.linear(o_l.to(dtype), proj_w.to(dtype), proj_b.to(dtype))


def sla_forward(q, k, v, proj_w, proj_b, topk_ratio: float, blkq: int = 128, blkk: int = 64,
                dtype=torch.bfloat16, mode: str = "exact", lut: Optional[torch.Tensor] = None) -> torch.Tensor:
    """SageSparseLinearAttention.forward (SLA/core.py:168-257) / SparseLinearAttention.forward (:81-119).
    q,k,v [B,L,H,D] (callers' layout, :181-183).  mode:
       'exact'  fp32 sparse attention + fp32 linear branch (the accuracy target)
       'triton' the bf16 Triton path's rounding points (P->dtype, o_s->dtype, linear branch in dtype)
       'sage'   INT8 Q/K emulation, P->dtype (unpinned)
    Returns [B,L,H,D] in q.dtype."""
    in_dtype = q.dtype
    qh, kh, vh = (t.transpose(1, 2).contiguous() for t in (q, k, v))
    if lut is None:
        _, lut, _ = get_block_map(qh, kh, topk_ratio, blkq, blkk)
    qh, kh, vh = qh.to(dtype), kh.to(dtype), vh.to(dtype)
    if mode == "exact":
        o_s = sparse_attention(qh, kh, vh, lut, blkq, blkk)
        o_l = linear_branch(qh, kh, vh, proj_w, proj_b, dtype, exact=True)
        o = o_s + o_l
    elif mode == "triton":
        o_s = sparse_attention(qh, kh, vh, lut, blkq, blkk, p_dtype=dtype).to(dtype)
        o_l = linear_branch(qh, kh, vh, proj_w, proj_b, dtype, exact=False)
        o = o_s + o_l
    elif mode == "sage":
        q_i8, q_s, k_i8, k_s, _ = sage_quant_qk(qh, kh, blkq, blkk)
        o_s = sparse_attention(qh, kh, vh, lut, blkq, blkk, p_dtype=dtype, q_i8=q_i8, q_s=q_s, k_i8=k_i8, k_s=k_s)
        o_l = linear_branch(qh, kh, vh, proj_w, proj_b, dtype, exact=True)
        o = o_s + o_l
    else:
        raise ValueError(mode)
    return o.to(in_dtype).transpose(1, 2).contiguous()


def sla_forward_block(q, k, v, proj_w, proj_b, head: int, m_blk: int, ids: torch.Tensor, blkq: int = 128, blkk: int = 64,
                      dtype=torch.bfloat16, mode: str = "exact", feature_map: str = "softmax",
                      batch: int = 0) -> torch.Tensor:
    """sla_forward restricted to ONE query block of ONE head (full-size parity sampling: the whole tensor would take the
    CPU minutes).  q,k,v [B,L,H,D]; `ids` = the selected key-block ids of that query block.  Same arithmetic and modes as
    sla_forward (SLA/core.py:168-257): the key mean, the K quantisation and the linear-attention moments still run over
    all L keys of the head.  Returns [rows, D] in q.dtype."""
    in_dtype = q.dtype
    l, d = q.shape[1], q.shape[3]
    r0, r1 = m_blk * blkq, min(l, (m_blk + 1) * blkq)
    qh = q[batch, :, head].to(dtype)[None, None]          # [1,1,L,D]
    kh = k[batch, :, head].to(dtype)[None, None]
    vh = v[batch, :, head].to(dtype)[None, None]
    qb = qh[:, :, r0:r1]
    lut = ids.reshape(1, 1, 1, -1)
    if mode == "sage":
        arg_k, _ = smooth_k(kh)
        q_i8, q_s = sage_quant_blocks(qb, blkq)
        k_i8, k_s = sage_quant_blocks(arg_k, blkk)
        o_s = sparse_attention(qb, kh, vh, lut, blkq, blkk, p_dtype=dtype, q_i8=q_i8, q_s=q_s, k_i8=k_i8, k_s=k_s)
    elif mode == "triton":
        o_s = sparse_attention(qb, kh, vh, lut, blkq, blkk, p_dtype=dtype).to(dtype).float()
    else:
        o_s = sparse_attention(qb, kh, vh, lut, blkq, blkk)
    fq, fk = feature_maps(feature_map)
    pq = fq(qb.float()).to(dtype).float()
    pk = fk(kh.float()).to(dtype).float()
    kv = pk.transpose(-1, -2) @ vh.float()
    ks = pk.sum(-2, keepdim=True)
    o_l = (pq @ kv) / (1e-5 + (pq * ks).sum(-1, keepdim=True))
    o_l = o_l @ proj_w.float().t() + proj_b.float()
    return (o_s + o_l)[0, 0].to(in_dtype)


def feature_maps(name: str):
    """SLA/core.py:57-73: 'softmax' (over D), 'elu' (elu(x)+1), 'relu'."""
    if name == "softmax":
        return (lambda x: torch.softmax(x, -1)), (lambda x: torch.softmax(x, -1))
    if name == "elu":
        return (lambda x: F.elu(x) + 1), (lambda x: F.elu(x) + 1)
    if name == "relu":
        return F.relu, F.relu
    raise NotImplementedError(f"Not supported feature map {name}.")


# =============================================================================================
# LTX-2 prologue variants (config 5) — ltx_core/model/transformer/transformer.py:21-94, ltx_core/utils.py:7-12
# =============================================================================================
def ltx_rms_norm(x: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    return x * torch.rsqrt(x.float().pow(2).mean(-1, keepdim=True) + eps).to(x.dtype)


def ltx_row_quant_int8(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """ltx_distillation/tilelang_w8a8.py:16-36: scale = max(amax,1e-4)/127; round half away; clip [-128,127]."""
    xf = x.float()
    scale = xf.abs().amax(-1).clamp_min(1e-4) / 127.0
    y = xf / scale[:, None]
    r = torch.where(y >= 0, torch.floor(y + 0.5), torch.ceil(y - 0.5)).clamp_(-128, 127)
    return r.to(torch.int8), scale


def ltx_gemm_post_scale(a_q, a_s, b_q, b_s, bias, out_dtype=torch.bfloat16) -> torch.Tensor:
    """tilelang_w8a8.py:108-114: C = int32_acc * sA[i] * sB[j] + bias[j], cast to bf16.  As executed on the GPU: TileLang
    lowers the expression to `t = float(acc)*sA; u = t*sB; c = u + bias` and compiles it with nvcc's default -fmad, which
    contracts the last two into one FFMA (64 I2FP + 64 FMUL + 64 FFMA per thread in the SASS, no FADD; reproduced by
    tools/tilelang_epilogue_probe.py) -> c = fma(float(acc)*sA, sB, bias).  The fused multiply-add is evaluated in fp64
    (the product of two fp32 values is exact there) and rounded once to fp32."""
    acc = (a_q.double() @ b_q.double().t())                       # exact integer accumulation (|sum| < 2^53)
    t = acc.float() * a_s[:, None]                                # I2FP (round to nearest), FMUL
    b = torch.zeros(b_s.shape[0], dtype=torch.float64) if bias is None else bias.double()
    y = (t.double() * b_s.double()[None, :] + b[None, :]).float()  # FFMA
    return y.to(out_dtype)


# =============================================================================================
# One Wan DiT block's self-attention + FFN hot path (for bench cpu_baseline / block parity), wan2pt1.py:390-417
# =============================================================================================
def wan_block_forward(sd: dict, x: torch.Tensor, e0: torch.Tensor, angles: torch.Tensor, context: torch.Tensor,
                      dim: int, heads: int, eps: float = 1e-6, topk: float = 0.1, sla_mode: str = "exact",
                      lut: Optional[torch.Tensor] = None) -> torch.Tensor:
    """WanAttentionBlock.forward (rcm/networks/wan2pt1.py:390-417) after TurboDiffusion's model surgery
    (inference/modify_model.py:40-81), on CPU tensors.  `sd`: reference state-dict keys relative to blocks.<i>.
    x [L, dim], e0 [6, dim] fp32, angles [L, head_dim/2], context [Lc, dim].  `lut` [1, heads, Mblk, topk]: the key blocks
    the self-attention attends to (default: the oracle's own top-k selection)."""
    d = dim // heads
    l = x.shape[0]

    def lin(t, name, gelu=False):
        y = int8_linear(t, sd[name + ".int8_weight"], sd[name + ".scale"], sd[name + ".bias"])
        return F.gelu(y, approximate="tanh") if gelu else y

    e = (sd["modulation"][0] + e0).float()
    hmod = ln_modulate(x, e[1], e[0], eps)
    q = fast_rmsnorm(lin(hmod, "self_attn.q"), sd["self_attn.norm_q.weight"], eps).view(l, heads, d)
    k = fast_rmsnorm(lin(hmod, "self_attn.k"), sd["self_attn.norm_k.weight"], eps).view(l, heads, d)
    v = lin(hmod, "self_attn.v").view(l, heads, d)
    q, k = rope_interleaved(q, angles), rope_interleaved(k, angles)
    a = sla_forward(q[None], k[None], v[None], sd["self_attn.attn_op.local_attn.proj_l.weight"],
                    sd["self_attn.attn_op.local_attn.proj_l.bias"], topk, mode=sla_mode, lut=lut)[0].reshape(l, dim)
    x = gate_residual(x, lin(a, "self_attn.o"), e[2])
    hn = fast_layernorm(x, sd["norm3.weight"], sd["norm3.bias"], eps)
    cq = fast_rmsnorm(lin(hn, "cross_attn.q"), sd["cross_attn.norm_q.weight"], eps).view(1, l, heads, d)
    ck = fast_rmsnorm(lin(context, "cross_attn.k"), sd["cross_attn.norm_k.weight"], eps).view(1, -1, heads, d)
    cv = lin(context, "cross_attn.v").view(1, -1, heads, d)
    ca = dense_attention(cq.transpose(1, 2), ck.transpose(1, 2), cv.transpose(1, 2)).transpose(1, 2).reshape(l, dim)
    x = x + lin(ca, "cross_attn.o")
    hmod = ln_modulate(x, e[4], e[3], eps)
    y = lin(lin(hmod, "ffn.0", gelu=True), "ffn.2")
    return gate_residual(x, y, e[5])


def stats(a: torch.Tensor, b: torch.Tensor) -> dict:
    """Error summary used by the parity tests."""
    a, b = a.double().flatten(), b.double().flatten()
    diff = (a - b).abs()
    return {
        "max_abs": diff.max().item(),
        "rel_l2": (diff.norm() / b.norm().clamp_min(1e-30)).item(),
        "cos": (torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30)).item(),
    }
