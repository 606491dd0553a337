"""Mirror of turbodiffusion/SLA/core.py: SparseLinearAttention / SageSparseLinearAttention on B200.

Same constructor arguments, parameters (`proj_l`, fp32, zero-init) and call convention (q,k,v in [B, L, H, D], result in
the same layout and dtype; SLA/core.py:181-183,253).  The forward is five kernel launches:
  quant_qk (key mean, pooled means, INT8 Q / smoothed K)  ->  block_map (pooled score, top-k, LUT)
  -> linear_moments (phi(K)^T V, sum phi(K); split-L partials reduced in a fixed order)  ->  project_moments (proj_l folded
  into the moment matrix)
  -> attn_fwd (sparse INT8 QK^T, softmax, PV, linear branch, merge).
Inputs are consumed in place in their [B, L, H, D] layout; no transposed copies of q/k/v are made.
"""
from __future__ import annotations

import ctypes
import functools
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from .._lib import DTYPE_TAG, check, lib, ptr, require_cuda, stream_ptr
from .utils import QKPrep, block_map_from_pools, get_block_map, get_cuda_arch, quant_qk  # noqa: F401

SAGESLA_ENABLED = True   # the INT8 path is built in (no SpargeAttn dependency)
SAGE2PP_ENABLED = True


FEATURE_TAG = {"softmax": 0, "elu": 1, "relu": 2}   # SLA/core.py:57-73


@functools.lru_cache(maxsize=256)
def moments_workspace_bytes(b: int, l: int, h: int, d: int) -> int:
    """Scratch bytes tdb200_sla_linear_moments_ws needs for k/v [b, l, h, d] (a function of the shape alone)."""
    n = ctypes.c_int64(0)
    check(lib().tdb200_sla_linear_moments_workspace(b, l, h, d, ctypes.byref(n)), "sla_linear_moments_workspace", launches=0)
    return n.value


def linear_moments(k: torch.Tensor, v: torch.Tensor, feature: int = 0):
    """kv [B,H,D(v),D(k)] fp32, ksum [B,H,D] fp32 of the local keys (accumulated: add shards / all-reduce).  D in {64, 128};
    `feature`: 0 softmax over D, 1 elu+1, 2 relu.  Bit-reproducible: the partial sums of the CTAs that split L are reduced
    in a fixed order."""
    b, l, h, d = k.shape
    buf = torch.zeros(b * h * d * (d + 1), dtype=torch.float32, device=k.device)        # one fill for both accumulators
    kv, ksum = buf[: b * h * d * d].view(b, h, d, d), buf[b * h * d * d:].view(b, h, d)
    nbytes = moments_workspace_bytes(b, l, h, d)
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=k.device)
    check(lib().tdb200_sla_linear_moments_ws(ptr(k), ptr(v), DTYPE_TAG[k.dtype], b, l, h, d, feature, ptr(kv), ptr(ksum),
                                             ptr(ws), nbytes, stream_ptr(k.device)), "sla_linear_moments")
    return kv, ksum


def project_moments(proj_w: torch.Tensor, kv: torch.Tensor, dtype) -> torch.Tensor:
    """kvw [B,H,D_out,D_k] = T(proj_w . kv): proj_l's weight folded into the moment matrix (the fused kernel's last MMA)."""
    b, h, d, _ = kv.shape
    w = proj_w if (proj_w.dtype == torch.float32 and proj_w.is_contiguous()) else proj_w.float().contiguous()
    assert kv.dtype == torch.float32 and kv.is_contiguous() and w.shape == (d, d)
    out = torch.empty(b, h, d, d, dtype=dtype, device=kv.device)
    check(lib().tdb200_sla_project_moments(ptr(w), ptr(kv), DTYPE_TAG[dtype], b * h, d, ptr(out), stream_ptr(kv.device)),
          "sla_project_moments")
    return out


ATTN_IMPL = os.environ.get("TDB200_ATTN_IMPL", "v1")  # "v1": one CTA per query block; "v2": persistent kernel (measured slower, see DESIGN)


ATTN_TIMER = None  # bench.py installs a callable(h, mblk, topk, d) -> context manager to time the fused-attention launches


def attn_fwd(prep, v, q, lut, topk, kvw, ksum, proj_b, sm_scale, lk=None, impl=None, feature=0):
    if ATTN_TIMER is not None:
        with ATTN_TIMER(q.shape[2] * q.shape[0], (q.shape[1] + 127) // 128, topk, q.shape[3]):
            return _attn_fwd(prep, v, q, lut, topk, kvw, ksum, proj_b, sm_scale, lk, impl, feature)
    return _attn_fwd(prep, v, q, lut, topk, kvw, ksum, proj_b, sm_scale, lk, impl, feature)


def _attn_fwd(prep, v, q, lut, topk, kvw, ksum, proj_b, sm_scale, lk=None, impl=None, feature=0):
    b, l, h, d = q.shape
    lk = v.shape[1] if lk is None else lk
    out = torch.empty_like(q)
    if getattr(prep, "k_seq_major", False):   # INT8 K in the gathered [B, Lk, H, D] layout (dist.py)
        if d != 128 or feature != 0:
            raise NotImplementedError("sequence-major INT8 K is served by the 128-wide softmax kernel only")
        check(lib().tdb200_sla_attn_fwd_kseq(ptr(prep.q_i8), ptr(prep.q_scale), ptr(prep.k_i8), ptr(prep.k_scale), ptr(v),
                                             ptr(q), DTYPE_TAG[q.dtype], ptr(lut), topk, ptr(kvw), ptr(ksum), ptr(proj_b),
                                             ptr(out), b, l, lk, h, d, float(sm_scale), stream_ptr(q.device)), "sla_attn_fwd")
    elif (impl or ATTN_IMPL) == "v1" and d == 128 and feature == 0:
        check(lib().tdb200_sla_attn_fwd(ptr(prep.q_i8), ptr(prep.q_scale), ptr(prep.k_i8), ptr(prep.k_scale), ptr(v),
                                        ptr(q), DTYPE_TAG[q.dtype], ptr(lut), topk, ptr(kvw), ptr(ksum), ptr(proj_b),
                                        ptr(out), b, l, lk, h, d, float(sm_scale), stream_ptr(q.device)), "sla_attn_fwd")
    else:
        check(lib().tdb200_sla_attn_fwd_v2(ptr(prep.q_i8), ptr(prep.q_scale), ptr(prep.k_i8), ptr(prep.k_scale), ptr(v),
                                           ptr(q), DTYPE_TAG[q.dtype], ptr(lut), topk, ptr(kvw), ptr(ksum), ptr(proj_b),
                                           ptr(out), b, l, lk, h, d, float(sm_scale), feature, stream_ptr(q.device)),
              "sla_attn_fwd")
    return out


def attn_fwd_qk16(q, k, v, lut, topk, kvw, ksum, proj_b, sm_scale, lk=None):
    """The non-quantised sparse attention (a9', SLA/kernel.py:33-82): 16-bit Q.K^T on the tensor cores, fp32 scores."""
    b, l, h, d = q.shape
    lk = v.shape[1] if lk is None else lk
    out = torch.empty_like(q)
    check(lib().tdb200_sla_attn_fwd_qk16(ptr(q), ptr(k), ptr(v), DTYPE_TAG[q.dtype], ptr(lut), topk, ptr(kvw), ptr(ksum),
                                         ptr(proj_b), ptr(out), b, l, lk, h, d, float(sm_scale), stream_ptr(q.device)),
          "sla_attn_fwd_qk16")
    return out


class _SLABase(nn.Module):
    quantised_qk = True   # SageSparseLinearAttention: INT8 Q.K^T; SparseLinearAttention: 16-bit Q.K^T (128-wide heads)

    def __init__(self, head_dim, topk, feature_map="softmax", use_bf16=True, tie_feature_map_qk=True):
        super().__init__()
        self.dtype = torch.bfloat16 if use_bf16 else torch.float16
        self.topk = topk
        self.proj_l = nn.Linear(head_dim, head_dim, dtype=torch.float32)
        if feature_map == "elu":            # SLA/core.py:57-61
            self.feature_map_q = self.feature_map_k = lambda x: F.elu(x) + 1
        elif feature_map == "relu":         # :62-64
            self.feature_map_q = self.feature_map_k = nn.ReLU()
        elif feature_map == "softmax":      # :65-69
            self.feature_map_q = self.feature_map_k = lambda x: F.softmax(x, dim=-1)
        else:
            raise NotImplementedError(f"Not supported feature map {feature_map}.")
        self.feature = FEATURE_TAG[feature_map]   # evaluated inside the fused kernels (moments + attention epilogue)
        self.init_weights_()

    def init_weights_(self):
        with torch.no_grad():
            nn.init.zeros_(self.proj_l.weight)
            nn.init.zeros_(self.proj_l.bias)

    def forward(self, q, k, v, return_sparsity=False):
        """q,k,v [B, L, H, D] (any float dtype), D in {64, 128} (SLA/core.py:207) -> [B, L, H, D] in q.dtype."""
        require_cuda(q, k, v)
        dtype = q.dtype
        q, k, v = (t if (t.dtype == self.dtype and t.is_contiguous()) else t.to(self.dtype).contiguous() for t in (q, k, v))
        b, l, h, d = q.shape
        if d not in (64, 128):
            raise AssertionError("headdim should be in [64, 128].")  # SLA/core.py:207
        prep = quant_qk(q, k)
        nblk = prep.nblk
        real_topk = min(nblk, int(self.topk * nblk))
        if real_topk < 1:
            # the reference would select zero key blocks here (an empty softmax); short sequences get one block instead
            real_topk = 1
        sparse_map, lut = block_map_from_pools(prep.q_pool, prep.k_pool, real_topk)
        if getattr(self, "_keep_selection", None) is not None:
            self._keep_selection.update(lut=lut, sparse_map=sparse_map, topk=real_topk)
        kv, ksum = linear_moments(k, v, self.feature)
        # proj_l folded into the moments: (phi(q) KV / den) W^T + b == phi(q) (W KV^T)^T / den + b ; kv is [dv, dk]
        kvw = project_moments(self.proj_l.weight, kv, self.dtype)  # [B,H,d_out,d_k]
        # 128-wide heads with the softmax map run the one-CTA-per-query-block kernel (faster); 64-wide heads and the
        # elu / relu maps run the persistent kernel, which has native 64-wide tiles and the feature-map switch
        impl = ATTN_IMPL if (d == 128 and self.feature == 0) else "v2"
        if not self.quantised_qk and d == 128 and self.feature == 0:
            o = attn_fwd_qk16(q, k, v, lut, real_topk, kvw, ksum, self.proj_l.bias.float().contiguous(), d ** -0.5)
        else:
            o = attn_fwd(prep, v, q, lut, real_topk, kvw, ksum, self.proj_l.bias.float().contiguous(), d ** -0.5, impl=impl,
                         feature=self.feature)
        o = o if o.dtype == dtype else o.to(dtype)
        return (o, real_topk / nblk) if return_sparsity else o

    def forward_with_lut(self, q, k, v):
        """forward() that also returns the block selection it used: (o, {"lut": int32 [B,H,Mblk,topk] ascending key-block
        ids, "sparse_map": int8 [B,H,Mblk,Nblk], "topk": int}).  Test/diagnostic entry point (sampled oracle parity at
        full shapes needs the kernel's own selection)."""
        self._keep_selection = {}
        try:
            o = self.forward(q, k, v)
            return o, self._keep_selection
        finally:
            self._keep_selection = None


class SparseLinearAttention(_SLABase):
    """SLA/core.py:38-119: the non-quantised variant (`--attention_type sla`).  128-wide heads with the softmax feature map run
    the fused kernel with a 16-bit Q.K^T (the arithmetic of the reference's Triton _attn_fwd, SLA/kernel.py:33-82); 64-wide
    heads and the elu / relu maps are served by the INT8-QK kernel.  Block sizes are BLKQ=128, BLKK=64 (the configuration
    modify_model.py:50 requests); other values are accepted for signature compatibility with a warning."""
    quantised_qk = False

    def __init__(self, head_dim, topk, feature_map="softmax", BLKQ=64, BLKK=64, use_bf16=True, tie_feature_map_qk=True):
        super().__init__(head_dim, topk, feature_map, use_bf16, tie_feature_map_qk)
        self.BLKQ, self.BLKK = BLKQ, BLKK
        if (BLKQ, BLKK) != (128, 64):
            import warnings
            warnings.warn(f"SparseLinearAttention(BLKQ={BLKQ}, BLKK={BLKK}): the B200 kernels use 128-row query blocks and "
                          "64-row key blocks (the configuration TurboDiffusion's modify_model.py:50 requests); block "
                          "selection differs from the reference for other sizes", stacklevel=2)


class SageSparseLinearAttention(_SLABase):
    """SLA/core.py:122-257."""

    def __init__(self, head_dim, topk, feature_map="softmax", use_bf16=True, tie_feature_map_qk=True):
        super().__init__(head_dim, topk, feature_map, use_bf16, tie_feature_map_qk)


# ------------------------------------------------------------------------------------------------------------------------
# Names the LTX-2 client reaches for inside `SLA.core` (TurboT2AV ltx_distillation/acceleration.py:260-383,
# LTXSageSLAAttention._sparse_only_forward, the default path while proj_l is still zero): SpargeAttn's quantiser, LUT
# builder, V preparation and the Sage2++ kernel entry.  Here they are thin adapters onto the same C-ABI kernels the modules
# use; the tensors SpargeAttn would transform (transposed / padded / fp8 V) are carried by reference instead, because the
# fused kernel consumes 16-bit V in its original layout.
# ------------------------------------------------------------------------------------------------------------------------
def get_vanilla_qk_quant(q, k, km=None, BLKQ=128, BLKK=64):
    """q,k [B,H,L,D] -> (q_int8 [B,H,L,D], q_scale [B,H,Mblk], k_int8 of (k - mean_L k), k_scale [B,H,Nblk]); call site
    SLA/core.py:200-203.  `km` is accepted for signature compatibility (the key mean is recomputed by the fused prepass)."""
    if (BLKQ, BLKK) != (128, 64):
        raise NotImplementedError("the B200 path implements the non-sm90 block sizes (BLKQ=128, BLKK=64)")
    prep = quant_qk(q.transpose(1, 2).contiguous(), k.transpose(1, 2).contiguous())
    return prep.q_i8, prep.q_scale, prep.k_i8, prep.k_scale


def block_map_lut_triton(sparse_map):
    """sparse_map int8 [B,H,Mblk,Nblk] -> (lut int32 [B,H,Mblk,topk] ascending block ids, valid_block_num int32 [B,H,Mblk]).
    Maps produced by this package's get_block_map carry their LUT; others are rebuilt from the map (every row must select the
    same number of blocks, as get_block_map guarantees)."""
    valid = sparse_map.sum(-1, dtype=torch.int32)
    lut = getattr(sparse_map, "_tdb200_lut", None)
    if lut is None:
        b, h, m, n = sparse_map.shape
        topk = int(valid.reshape(-1)[0].item())
        lut = sparse_map.bool().nonzero()[:, -1].view(b, h, m, topk).to(torch.int32).contiguous()
    return lut, valid


class _FusedShim:
    """SpargeAttn `fused` namespace: V transposition / fp8 quantisation are not materialised; the outputs remember their source."""

    @staticmethod
    def transpose_pad_permute_cuda(v, out, tensor_layout=1):
        out._tdb200_src = v

    @staticmethod
    def scale_fuse_quant_cuda(v_in, v_fp8, v_scale, kv_len, scale_max=2.25, tensor_layout=1):
        v_fp8._tdb200_src = getattr(v_in, "_tdb200_src", v_in)


fused = _FusedShim()


def qk_int8_sv_f8_accum_f16_block_sparse_attn_inst_buf_fuse_v_scale_with_pv_threshold(
        q_int8, k_int8, v_fp8, o, lut, valid_block_num, pvthreshold, q_scale, k_scale, v_scale, tensor_layout=1,
        is_causal=False, qk_quant_gran=1, sm_scale=None, return_lse=0):
    """Sparse (softmax) branch only: o [B,H,L,D] <- block-sparse INT8-QK attention over the LUT's key blocks, the linear
    branch switched off (zero moments, zero bias).  Same kernel as SageSparseLinearAttention.forward."""
    v = getattr(v_fp8, "_tdb200_src", None)
    if v is None:
        raise RuntimeError("this adapter needs the 16-bit V that SLA.core.fused.* was called with")
    b, h, lq, d = q_int8.shape
    lk = k_int8.shape[2]
    prep = QKPrep()
    prep.q_i8, prep.q_scale, prep.k_i8, prep.k_scale = q_int8, q_scale, k_int8, k_scale
    prep.mblk, prep.nblk = (lq + 127) // 128, (lk + 63) // 64
    vt = v.transpose(1, 2).contiguous()                       # [B,L,H,D]
    qz = torch.zeros(b, lq, h, d, dtype=v.dtype, device=v.device)
    kvw = torch.zeros(b, h, d, d, dtype=v.dtype, device=v.device)
    ksum = torch.ones(b, h, d, dtype=torch.float32, device=v.device)
    pb = torch.zeros(d, dtype=torch.float32, device=v.device)
    out = attn_fwd(prep, vt, qz, lut, lut.shape[-1], kvw, ksum, pb, sm_scale if sm_scale is not None else d ** -0.5, lk=lk,
                   impl=None if d == 128 else "v2")
    o.copy_(out.transpose(1, 2))
    return o


class _QattnShim:
    """SpargeAttn's `qattn` extension module holds the sm80 / sm90 kernels; on B200 the client takes the Sage2++ entry above."""

    def __getattr__(self, name):
        raise NotImplementedError(f"SLA.core.qattn.{name}: sm80/sm90 SpargeAttn kernels have no B200 counterpart; "
                                  "get_cuda_arch() reports sm100, which routes callers to the fused kernel")


qattn = _QattnShim()
