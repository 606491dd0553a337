"""Generate tests/golden/*.pt by running the REFERENCE's own code on CPU (this container only).

  TRITON_INTERPRET=1 python tools/make_golden.py [norm] [sla] [ltx]     (no names = all; each group reseeds itself)

Imports /root/reference/turbodiffusion (ops/core.py Triton norms, SLA/utils.py, SLA/kernel.py, SLA/core.py) with a stub
for the CUDA-only pybind module, runs the Triton kernels through Triton's CPU interpreter and stores small seeded
input/output pairs.  /root/reference does not exist on the GPU box, so only the fixtures travel.
"""
import os
import sys
import types

os.environ["TRITON_INTERPRET"] = "1"
REF = "/root/reference/turbodiffusion"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")

stub = types.ModuleType("turbo_diffusion_ops")
stub.quant_cuda = stub.gemm_cuda = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("CUDA-only"))
sys.modules["turbo_diffusion_ops"] = stub
sys.path.insert(0, REF)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import triton.language as tl  # noqa: E402
import triton.runtime.interpreter as _interp  # noqa: E402

# Triton's CPU interpreter truncates fp32 -> bf16 (cast_impl passes rounding_mode=None), whereas the compiled GPU kernel
# emits cvt.rn.bf16.f32 (round to nearest even).  Patch that one conversion so the goldens carry the GPU semantics.
_orig_convert = _interp._convert_float


def _convert_float_rne(inp, in_dtype, out_dtype, rounding_mode):
    if in_dtype == tl.float32 and out_dtype == tl.bfloat16:
        t = torch.from_numpy(np.ascontiguousarray(inp).view(np.float32).copy()).to(torch.bfloat16)
        return t.view(torch.int16).numpy().view(np.uint16).reshape(inp.shape)
    return _orig_convert(inp, in_dtype, out_dtype, rounding_mode)


_interp._convert_float = _convert_float_rne

# The interpreter stores bf16 as uint16 and its create_dot() feeds those raw bit patterns to np.matmul.  Upcast bf16
# operands to fp32 first: products of bf16 values are exact in fp32 and the GPU accumulates in fp32 as well.
_orig_dot = _interp.InterpreterBuilder.create_dot


def _bf16_bits_to_f32(a):
    return (a.astype(np.uint32) << 16).view(np.float32)


def _create_dot(self, a, b, d, input_precision, max_num_imprecise_acc):
    if a.dtype == tl.bfloat16 or b.dtype == tl.bfloat16:
        a_data = _bf16_bits_to_f32(a.data) if a.dtype == tl.bfloat16 else a.data.astype(np.float32)
        b_data = _bf16_bits_to_f32(b.data) if b.dtype == tl.bfloat16 else b.data.astype(np.float32)
        return _interp.TensorHandle(np.matmul(a_data, b_data, dtype=d.data.dtype) + d.data, d.dtype.scalar)
    return _orig_dot(self, a, b, d, input_precision, max_num_imprecise_acc)


_interp.InterpreterBuilder.create_dot = _create_dot

import ops.core as ref_ops  # noqa: E402
import SLA.utils as ref_utils  # noqa: E402
import SLA.core as ref_sla  # noqa: E402

# SLA/core.py:116 enters torch.amp.autocast('cuda', dtype) around proj_l; on CPU tensors that context is a no-op, so
# redirect it to the CPU autocast to get the same bf16 evaluation of the fp32 Linear the GPU run performs.
_orig_autocast = torch.amp.autocast
torch.amp.autocast = lambda device_type, dtype=None, **kw: _orig_autocast("cpu", dtype=dtype, **kw)

os.makedirs(OUT, exist_ok=True)
torch.manual_seed(20260922)
ONLY = set(sys.argv[1:])


def want(group):
    return not ONLY or group in ONLY



def save(name, **kw):
    torch.save(kw, os.path.join(OUT, name + ".pt"))
    print("wrote", name, {k: (tuple(v.shape), str(v.dtype)) if torch.is_tensor(v) else v for k, v in kw.items()})


# ---- norms (ops/core.py Triton kernels), N not a power of two exposes the variance padding behaviour
for n in ((1536, 5120, 256) if want("norm") else ()):
    rows = 32 if n <= 512 else 6  # the reference kernels do not mask rows when N <= 512 (BLOCK_M = 32): keep M % 32 == 0
    x = (torch.randn(rows, n) * 1.3 + 0.8).bfloat16()
    w = torch.rand(n) + 0.5
    b = torch.randn(n) * 0.1
    rms = ref_ops.rmsnorm(x.float(), w, 1e-6).to(x.dtype)                       # FastRMSNorm.forward
    ln = ref_ops.layernorm(x.float(), None, None, 1e-6, False).to(x.dtype)      # FastLayerNorm.forward (no affine)
    ln_aff = ref_ops.layernorm(x.float(), w, b, 1e-6, True).to(x.dtype)
    ln_f32 = ref_ops.layernorm(x.float(), None, None, 1e-6, False)
    save(f"norm_n{n}", x=x, w=w, b=b, rms=rms, ln=ln, ln_aff=ln_aff, ln_f32=ln_f32, eps=1e-6)

# ---- block map + Triton sparse attention + full SparseLinearAttention.forward
for tag, (bsz, h, l, d, topk) in ({"sla_a": (1, 2, 600, 128, 0.25), "sla_b": (2, 1, 333, 64, 0.5)}.items() if want("sla") else ()):
    q = torch.randn(bsz, l, h, d).bfloat16()
    k = (torch.randn(bsz, l, h, d) + torch.randn(1, 1, h, d) * 2.0).bfloat16()  # per-channel key bias: smooth-K matters
    v = torch.randn(bsz, l, h, d).bfloat16()
    qh, kh = q.transpose(1, 2).contiguous(), k.transpose(1, 2).contiguous()
    pooled_q = ref_utils.mean_pool(qh, 128)
    arg_k = kh - torch.mean(kh, dim=-2, keepdim=True)
    pooled_k = ref_utils.mean_pool(arg_k, 64)
    score = pooled_q @ pooled_k.transpose(-1, -2)
    sparse_map, lut, real_topk = ref_utils.get_block_map(qh, kh, topk_ratio=topk, BLKQ=128, BLKK=64)
    mod = ref_sla.SparseLinearAttention(d, topk, BLKQ=128, BLKK=64)
    with torch.no_grad():
        mod.proj_l.weight.copy_(torch.randn(d, d) * 0.05)
        mod.proj_l.bias.copy_(torch.randn(d) * 0.05)
        out = mod(q, k, v)
        o_s = ref_sla._attention.apply(qh, kh, v.transpose(1, 2).contiguous(), sparse_map, lut, real_topk, 128, 64)
    # sla_a's inputs would take the file past 1 MB: oracle/golden.py draws them again and checks this checksum instead
    inputs = dict(checksum=torch.stack([t.view(torch.int16).to(torch.int64).sum() for t in (q, k, v)])) if tag == "sla_a" else \
        dict(q=q, k=k, v=v)
    save(tag, **inputs, pooled_q=pooled_q, pooled_k=pooled_k, score=score, sparse_map=sparse_map, lut=lut,
         topk=real_topk, topk_ratio=topk, proj_w=mod.proj_l.weight.detach().clone(),
         proj_b=mod.proj_l.bias.detach().clone(), o_s=o_s, out=out)

# ---- full-size block maps (Nblk = 512 for Wan-1.3B 480p, 1182 for Wan-14B 720p): the reference's own get_block_map on seeded
#      inputs.  q,k are NOT stored (tens of MB): the test regenerates them on the CPU from the same generator and checks
#      their checksum.  To stay under 1 MB the fixture holds the key mean and pooled keys of the kept heads and, for a seeded
#      sample of 64 query blocks (the first and the ragged last one always in), the pooled queries, the bf16 scores and the
#      selected key blocks as sorted indices.
def blockmap_inputs(l, h, d, seed):
    """Shared with tests/test_gpu_blockmap_golden.py (must stay byte-identical there)."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(1, h, l, d, generator=g).bfloat16()
    k = (torch.randn(1, h, l, d, generator=g) + torch.randn(1, h, 1, d, generator=g) * 2.0).bfloat16()
    return q, k


def blockmap_rows(nq, seed, n=64):
    pick = torch.randperm(nq, generator=torch.Generator().manual_seed(seed))[:n - 2]
    return torch.unique(torch.cat([pick, torch.tensor([0, nq - 1])]))


for tag, (l, h, d, topk, seed, heads) in ({"blockmap_n512": (32760, 2, 128, 0.1, 512, [0, 1]),
                                           "blockmap_n1182": (75600, 2, 128, 0.1, 1182, [0]),
                                           "blockmap_n512_d64": (32760, 2, 64, 0.15, 564, [0, 1])}.items()
                                          if want("blockmap") else ()):
    qh, kh = blockmap_inputs(l, h, d, seed)
    pooled_q = ref_utils.mean_pool(qh, 128)
    arg_k = kh - torch.mean(kh, dim=-2, keepdim=True)
    pooled_k = ref_utils.mean_pool(arg_k, 64)
    score = pooled_q @ pooled_k.transpose(-1, -2)
    sparse_map, lut, real_topk = ref_utils.get_block_map(qh, kh, topk_ratio=topk, BLKQ=128, BLKK=64)
    csum = torch.stack([qh.view(torch.int16).to(torch.int64).sum(), kh.view(torch.int16).to(torch.int64).sum()])
    rows, hs = blockmap_rows(pooled_q.shape[2], seed), torch.tensor(heads)
    sm = sparse_map[:, hs][:, :, rows].bool()
    sel = torch.sort(torch.topk(sm.float(), real_topk, -1).indices, -1).values.to(torch.int16)
    save(tag, l=l, h=h, d=d, seed=seed, checksum=csum, heads=heads, rows=rows, kmean=torch.mean(kh, dim=-2)[:, hs].clone(),
         pooled_q=pooled_q[:, hs][:, :, rows].clone(), pooled_k=pooled_k[:, hs].clone(),
         score=score[:, hs][:, :, rows].clone(), lut=sel, topk=real_topk, topk_ratio=topk)

# ---- LTX per-row INT8 quantisation (TurboT2AV ltx_distillation/tilelang_w8a8.py:16-36), the Triton kernel itself
if want("ltx"):
    import importlib.util
    torch.manual_seed(20260923)
    spec = importlib.util.spec_from_file_location(
        "ref_tilelang_w8a8", "/root/reference/TurboT2AV/LTX-2/packages/ltx-distillation/src/ltx_distillation/tilelang_w8a8.py")
    ref_tl = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_tl)
    import triton
    for k in (384, 4096):
        m = 12
        x = (torch.randn(m, k) * 1.7).bfloat16()
        x[:, ::97] *= 9.0                       # outlier columns
        x[3] = 0                                # amax below the 1e-4 floor
        x[4] = x[4].abs().clamp_min(0.01)       # all positive
        x[5, :8] = torch.tensor([127.0, 63.5, -63.5, 0.5, -0.5, 1.5, -1.5, 2.5]).bfloat16()   # exact .5 ties at scale 1
        x[5, 8:] = x[5, 8:].clamp(-100, 100)
        q = torch.empty(m, k, dtype=torch.int8)
        sc = torch.empty(m, dtype=torch.float32)
        ref_tl._row_quant_kernel[(m,)](x, q, sc, k, triton.next_power_of_2(k))     # body of row_quant_int8 (:39-52)
        save(f"ltx_rowquant_k{k}", x=x, q=q, s=sc)
