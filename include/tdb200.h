/*
 * tdb200.h — C ABI of libtdb200.so: the B200 (sm_100a) implementation of TurboDiffusion's denoise hot path.
 *
 * This is the drop-in boundary.  Every entry point replaces one interface of the reference
 * (thu-ml/TurboDiffusion; citations are file:line inside that repository):
 *
 *   turbo_diffusion_ops.quant_cuda        turbodiffusion/ops/quant/quant.cu:28-71     -> tdb200_quant_int8_block128
 *   turbo_diffusion_ops.gemm_cuda         turbodiffusion/ops/gemm/gemm.cu:27-68       -> tdb200_gemm_w8a8
 *   turbo_diffusion_ops.rms_norm_cuda     turbodiffusion/ops/norm/rmsnorm.cu:57-59    -> tdb200_rms_norm_f32
 *   turbo_diffusion_ops.layer_norm_cuda   turbodiffusion/ops/norm/layernorm.cu:60-62  -> tdb200_layer_norm_f32
 *   ops.FastRMSNorm / FastLayerNorm fwd   turbodiffusion/ops/core.py:441-442,477-478  -> tdb200_rms_norm / tdb200_layer_norm
 *   AdaLN modulate / gate (caller math)   turbodiffusion/rcm/networks/wan2pt1.py:398-417 -> tdb200_layer_norm_modulate[_quant], tdb200_gate_residual
 *   rope_apply                            turbodiffusion/rcm/networks/wan2pt1.py:156-178 -> tdb200_rope_interleaved, tdb200_rms_norm_rope
 *   SLA.utils.get_block_map               turbodiffusion/SLA/utils.py:55-67           -> tdb200_sla_block_map
 *   spas_sage_attn get_vanilla_qk_quant   call site turbodiffusion/SLA/core.py:200-203 -> tdb200_sla_quant_qk
 *   Sage block-sparse attention + linear  turbodiffusion/SLA/core.py:231-253          -> tdb200_sla_linear_moments, tdb200_sla_attn_fwd
 *
 * Conventions
 *   - plain pointers and sizes; all pointers are DEVICE pointers unless stated; no allocation inside;
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns without synchronising;
 *   - return value: TDB200_OK or a negative TDB200_ERR_* code; the library never calls exit();
 *     tdb200_last_error() returns a thread-local description of the last failure;
 *   - reentrant per stream; no internal threads, no global mutable state besides per-device caches;
 *   - 16-bit floating tensors are described by a TDB200_DTYPE_* tag.
 */
#ifndef TDB200_H_
#define TDB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TDB200_ABI_VERSION 1

#define TDB200_OK 0
#define TDB200_ERR_INVALID_ARG (-1)  /* null pointer, bad size, misaligned buffer            */
#define TDB200_ERR_UNSUPPORTED (-2)  /* shape/dtype outside what the kernels implement        */
#define TDB200_ERR_CUDA (-3)         /* a CUDA runtime/driver call failed (see last_error)    */
#define TDB200_ERR_ARCH (-4)         /* current device is not compute capability 10.x         */
#define TDB200_ERR_WORKSPACE (-5)    /* caller-provided workspace too small                   */

#define TDB200_DTYPE_BF16 0
#define TDB200_DTYPE_FP16 1

/* ABI version of the loaded library (== TDB200_ABI_VERSION it was built with). */
int tdb200_abi_version(void);
/* Thread-local, NUL-terminated description of the most recent error on this thread ("" if none). */
const char* tdb200_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * a1. per-128x128-block symmetric INT8 quantisation   (ops/quant/quant.hpp:86-99,122-164)
 *   x [m,k] row-major contiguous 16-bit float; q [m,k] int8; s [ceil(m/128), ceil(k/128)] fp32 row-major.
 *   per block: amax = max(1e-8, max|x|); s = amax/128; q = sat_s8(rint(x * (128/amax))).
 *   k must be a multiple of 8.  x and q 16-byte aligned.
 * ------------------------------------------------------------------------------------------- */
int tdb200_quant_int8_block128(const void* x, int x_dtype, int64_t m, int64_t k, int8_t* q, float* s, void* stream);
/* (q, s) = quant_int8_block128( T( gelu_tanh(x) ) ): the FFN activation (nn.GELU(approximate="tanh"),
 * rcm/networks/wan2pt1.py:375) and the quantisation of the down-projection's input in one HBM pass (2 B read, 1 B written
 * per element).  gelu in fp32 with one rounding to T, like torch on a 16-bit tensor. */
int tdb200_gelu_quant_int8_block128(const void* x, int x_dtype, int64_t m, int64_t k, int8_t* q, float* s, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a2. W8A8 GEMM with per-128-K-block rescale   (ops/gemm/kernel.hpp:391-427, utils.hpp:116-121)
 *   c[i,j] = T( sum_kb float(sum_{t in kb} a_q[i,t]*b_q[j,t]) * (a_s[i/128,kb]*b_s[j/128,kb]) )   fp32 FMA, kb ascending
 *   then, if bias != NULL,  c[i,j] = T(float(c[i,j]) + float(bias[j]))      (ops/core.py:410-411)
 *   a_q [m,k] int8, a_s [ceil(m/128), k/128]; b_q [n,k] int8 ("TN": both K-major), b_s [ceil(n/128), k/128];
 *   bias [n] of dtype c_dtype or NULL; c [m,n] row-major of dtype c_dtype.
 *   Requires k % 128 == 0 and n % 8 == 0 (the reference silently skips such shapes, gemm/launch.hpp:34-35;
 *   here they return TDB200_ERR_UNSUPPORTED).  tcgen05 kind::i8, TMA-staged tiles, accumulators in TMEM.
 * ------------------------------------------------------------------------------------------- */
int tdb200_gemm_w8a8(const int8_t* a_q, const float* a_s, const int8_t* b_q, const float* b_s, const void* bias,
                     void* c, int c_dtype, int64_t m, int64_t n, int64_t k, void* stream);
/* Same GEMM with a fused activation on the output:  TDB200_EPILOGUE_GELU_TANH computes
 * c = T(gelu_tanh(float(c_plain))) where c_plain is the value tdb200_gemm_w8a8 would store
 * (nn.GELU(approximate="tanh") after the FFN up-projection, rcm/networks/wan2pt1.py:375). */
#define TDB200_EPILOGUE_NONE 0
#define TDB200_EPILOGUE_GELU_TANH 1
int tdb200_gemm_w8a8_ex(const int8_t* a_q, const float* a_s, const int8_t* b_q, const float* b_s, const void* bias,
                        void* c, int c_dtype, int64_t m, int64_t n, int64_t k, int epilogue, void* stream);
/* One W8A8 GEMM for projections that share their input (the q/k/v of a self-attention; reference: the fused to_qkv / to_kv
 * packing of TurboT2AV ltx_distillation/acceleration.py:836-860): b_q [n,k], b_s and bias are the row-wise concatenation of
 * `parts` equal projections (n = parts * n_part, n_part a multiple of 256); c receives `parts` separate contiguous
 * [m, n_part] matrices.  Scales are per 128 weight rows, so every output equals tdb200_gemm_w8a8 on its own weights. */
int tdb200_gemm_w8a8_split(const int8_t* a_q, const float* a_s, const int8_t* b_q, const float* b_s, const void* bias,
                           void* c, int c_dtype, int64_t m, int64_t n, int64_t k, int64_t parts, void* stream);
/* GEMM whose output is emitted already block-quantised for the next W8A8 GEMM:
 *   (out_q, out_s) == tdb200_quant_int8_block128( output of tdb200_gemm_w8a8_ex in dtype `mid_dtype` )   bit for bit,
 * without the 16-bit tensor ever reaching HBM (FFN: Linear -> GELU -> Int8Linear, ops/core.py:28-57 called twice).
 * out_q [m,n] int8, out_s [ceil(m/128), n/128] fp32; n % 128 == 0. */
int tdb200_gemm_w8a8_quant_out(const int8_t* a_q, const float* a_s, const int8_t* b_q, const float* b_s,
                               const void* bias, int8_t* out_q, float* out_s, int mid_dtype, int64_t m, int64_t n,
                               int64_t k, int epilogue, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a3/a4. FastNorm
 *   *_f32 : the registered-but-unused reference entry points (fp32 in, fp32 out), 1 CTA per row.
 *   16-bit variants: the whole FastRMSNorm.forward / FastLayerNorm.forward including the caller-side
 *   casts (x.float() in, .to(x.dtype) out) in ONE pass: y = T(float(x) * rstd * w), etc.
 *   w / b are fp32 [n] or NULL (no affine).  n % 8 == 0 (16-bit) / n % 4 == 0 (fp32), n <= 16384.
 * ------------------------------------------------------------------------------------------- */
int tdb200_rms_norm_f32(const float* x, const float* w, float* y, int64_t m, int64_t n, float eps, void* stream);
int tdb200_layer_norm_f32(const float* x, const float* w, const float* b, float* y, int64_t m, int64_t n, float eps,
                          void* stream);
int tdb200_rms_norm(const void* x, int dtype, const float* w, void* y, int64_t m, int64_t n, float eps, void* stream);
int tdb200_layer_norm(const void* x, int dtype, const float* w, const float* b, void* y, int64_t m, int64_t n,
                      float eps, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a5. AdaLN prologue / epilogue   (rcm/networks/wan2pt1.py:398-417)
 *   layer_norm_modulate:        y = T( float(T(LN(x))) * (1 + scale[j]) + shift[j] )
 *   layer_norm_modulate_quant:  same value, emitted directly as a1-format int8 + block scales
 *                               (one stats pass + one tile pass instead of LN, 2 casts, modulate, quant).
 *                               row_stats: workspace of 2*m floats (mean, rstd per row).
 *   gate_residual:              out = T( x + T( y * T(gate[j]) ) )          (x + y*e under bf16 tensors)
 *   scale/shift/gate: fp32 [n] (one modulation vector: batch 1 per call).
 * ------------------------------------------------------------------------------------------- */
int tdb200_layer_norm_modulate(const void* x, int dtype, const float* scale, const float* shift, void* y, int64_t m,
                               int64_t n, float eps, void* stream);
int tdb200_layer_norm_modulate_quant(const void* x, int dtype, const float* scale, const float* shift, int8_t* q,
                                     float* s, float* row_stats, int64_t m, int64_t n, float eps, void* stream);
int tdb200_gate_residual(const void* x, const void* y, const float* gate, void* out, int dtype, int64_t m, int64_t n,
                         void* stream);
/* Cross-kernel fusion of the two above: the gate/residual update (gate == NULL: plain x + y) also emits the row
 * statistics (mean, rstd incl. the reference's variance padding term) of its OUTPUT, i.e. of the next LayerNorm's input,
 * and layer_norm_modulate_quant_stats is the tile pass alone, consuming them.  Results are bit-identical to
 * gate_residual followed by layer_norm_modulate_quant; one full read of the activation per LayerNorm is saved. */
int tdb200_gate_residual_stats(const void* x, const void* y, const float* gate, void* out, float* row_stats, int dtype,
                               int64_t m, int64_t n, float eps, void* stream);
int tdb200_layer_norm_modulate_quant_stats(const void* x, int dtype, const float* row_stats, const float* scale,
                                           const float* shift, int8_t* q, float* s, int64_t m, int64_t n, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a6. RoPE, interleaved pairs   (rcm/networks/wan2pt1.py:156-178; flash_attn interleaved=True)
 *   x, y [l, h, d] contiguous 16-bit; angles [l, d/2] fp32 (radians).
 *   y[2i] = T(x[2i]*cos - x[2i+1]*sin), y[2i+1] = T(x[2i]*sin + x[2i+1]*cos), math in fp32.
 *   rms_norm_rope: y = rope( T( rmsnorm_{over h*d}(x) * w ) ) in one pass (norm_q/norm_k + rope_apply).
 * ------------------------------------------------------------------------------------------- */
int tdb200_rope_interleaved(const void* x, int dtype, const float* angles, void* y, int64_t l, int64_t h, int64_t d,
                            void* stream);
int tdb200_rms_norm_rope(const void* x, int dtype, const float* w, const float* angles, void* y, int64_t l, int64_t h,
                         int64_t d, float eps, void* stream);
/* rms_norm_rope with the rotation read from a table cos_sin [l, d/2, 2] fp32 = (cos a, sin a) of the same angles (the reference
 * precomputes its complex `freqs` once per call as well, wan2pt1.py:111-137,156-178): one table serves every head, projection
 * and layer of a denoise step, and the kernel carries no range reduction / sin / cos work. */
int tdb200_rms_norm_rope_table(const void* x, int dtype, const float* w, const float* cos_sin, void* y, int64_t l, int64_t h,
                               int64_t d, float eps, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a7-a10. SLA / SageSLA.  q, k, v, out are [b, l, h, d] contiguous 16-bit (the layout the module is
 * called with, SLA/core.py:181-183), d in {64, 128}.  Block sizes: BLKQ = 128 query rows, BLKK = 64 key rows
 * (the non-sm90 branch, SLA/core.py:191-193).  mblk = ceil(l/128), nblk = ceil(l/64).
 *
 * tdb200_sla_quant_qk   one pass over q [b,lq,h,d] and two over k [b,lk,h,d] (lq != lk when the query rows are one rank's
 *     sequence shard and k is the gathered key slab; mblk = ceil(lq/128), nblk = ceil(lk/64)):
 *     kmean  [b,h,d]  fp32   = sum_l k / l  (T-rounded copy is what is subtracted, SLA/utils.py:56)
 *     q_i8   [b,h,l,d] int8, q_scale [b,h,mblk];  k_i8 [b,h,l,d] int8 of T(k - T(kmean)), k_scale [b,h,nblk]
 *                             scale = amax/127 + 1e-7, round half away from zero (SpargeAttn get_vanilla_qk_quant)
 *     q_pool [b,h,mblk,d] T,  k_pool [b,h,nblk,d] T   block means (SLA/utils.py:21-52; actual row count in the tail)
 *     q == NULL or k == NULL runs only the other half (the sequence-parallel path prepares Q while the K/V all-gather
 *     is still in flight).
 * tdb200_sla_block_map  pooled score T(q_pool . k_pool^T), top-`topk` per row (ties -> lowest index),
 *     sparse_map [b,h,mblk,nblk] int8 0/1 (SLA/utils.py:64-66) and lut [b,h,mblk,topk] int32 ascending block ids.
 * tdb200_sla_linear_moments   phi = softmax over d;  kv [b,h,d(v),d(k)] fp32 = sum_l v[l,:]^T phi(k)[l,:],
 *     ksum [b,h,d] fp32 = sum_l phi(k)[l,:]   (SLA/core.py:243-247).  Both must be zeroed by the caller
 *     (they are accumulated, so sequence shards can be summed with one all-reduce).  These two entry points add the
 *     partial sums of the CTAs that split l with fp32 atomics, in arrival order: the last bits vary from run to run.
 *     tdb200_sla_linear_moments_ws is the bit-reproducible form.
 * tdb200_sla_attn_fwd   o = T( sparse_softmax_attention(q_i8,k_i8,v; lut) + proj( phi(q) kv / (1e-5 + phi(q).ksum) ) )
 *     kvw [b,h,d(out),d(k)] T = (proj_w . kv) so that proj is folded into the moment matrix; proj_b [d] fp32.
 *     The int8 QK^T, online softmax (exp2), PV, linear branch and merge run in one tcgen05 kernel.
 * ------------------------------------------------------------------------------------------- */
int tdb200_sla_quant_qk(const void* q, const void* k, int dtype, int64_t b, int64_t lq, int64_t lk, int64_t h, int64_t d,
                        float* kmean, int8_t* q_i8, float* q_scale, int8_t* k_i8, float* k_scale, void* q_pool,
                        void* k_pool, void* stream);
int tdb200_sla_block_map(const void* q_pool, const void* k_pool, int dtype, int64_t b, int64_t h, int64_t mblk,
                         int64_t nblk, int64_t d, int64_t topk, int8_t* sparse_map, int32_t* lut, void* stream);
int tdb200_sla_linear_moments(const void* k, const void* v, int dtype, int64_t b, int64_t l, int64_t h, int64_t d,
                              float* kv, float* ksum, void* stream);
/* Same with the feature map of the linear branch selectable (0 softmax, 1 elu+1, 2 relu; SLA/core.py:57-73) and head dim
 * 64 or 128 (kv [b,h,d,d], ksum [b,h,d]). */
int tdb200_sla_linear_moments_ex(const void* k, const void* v, int dtype, int64_t b, int64_t l, int64_t h, int64_t d,
                                 int feature, float* kv, float* ksum, void* stream);
/* Bit-reproducible moments: kv += sum, ksum += sum (same meaning and arguments as _ex), with the split-l partial sums
 * stored to `workspace` and then reduced in a fixed order by a second kernel (2 launches).  The result depends on the inputs
 * and the shape only: the same on every run and every device.  workspace: device memory of at least the size
 * tdb200_sla_linear_moments_workspace reports for the shape (a host-side query, no CUDA call), 16-byte aligned, any
 * contents, not read by the caller; ksum 16-byte aligned.  A smaller workspace returns TDB200_ERR_WORKSPACE.
 * Calls that share one workspace must be ordered (the same stream). */
int tdb200_sla_linear_moments_workspace(int64_t b, int64_t l, int64_t h, int64_t d, int64_t* bytes);
int tdb200_sla_linear_moments_ws(const void* k, const void* v, int dtype, int64_t b, int64_t l, int64_t h, int64_t d,
                                 int feature, float* kv, float* ksum, void* workspace, int64_t workspace_bytes, void* stream);
/* kvw [bh,d,d] T = T(proj_w [d,d] . kv [bh,d,d]): folds proj_l's weight (SLA/core.py:246 `self.proj_l(o_l)`) into the moment
 * matrix so the fused kernel applies it with its last MMA; fp32 FMA chain over d_v. */
int tdb200_sla_project_moments(const float* proj_w, const float* kv, int dtype, int64_t bh, int64_t d, void* kvw, void* stream);
int tdb200_sla_attn_fwd(const int8_t* q_i8, const float* q_scale, const int8_t* k_i8, const float* k_scale,
                        const void* v, const void* q, int dtype, const int32_t* lut, int64_t topk, const void* kvw,
                        const float* ksum, const float* proj_b, void* out, int64_t b, int64_t l, int64_t lk,
                        int64_t h, int64_t d, float sm_scale, void* stream);
/* Sequence-parallel form of the key half of tdb200_sla_quant_qk (reference: the context-parallel attention of
 * rcm/utils/a2a_cp.py:66-182 exchanges 16-bit K; here each rank quantises its own key rows and the INT8 tensor travels).
 *   tdb200_sla_kmean_partial  partial [b,h,ceil(l/128),d] fp32 = column sums of each 128-row chunk of k [b,l,h,d];
 *   tdb200_sla_kmean_final    kmean [b,h,d] = (fixed-order sum of `chunks` partials) / l_total  -- the reduction
 *                             tdb200_sla_quant_qk runs, so gathering every rank's partials reproduces its mean bit for bit;
 *   tdb200_sla_quant_k_seq    smoothed Sage INT8 of k's rows: k_i8 in the INPUT layout [b,l,h,d], k_scale [b,h,ceil(l/64)],
 *                             k_pool [b,h,ceil(l/64),d];
 *   tdb200_sla_attn_fwd_kseq  tdb200_sla_attn_fwd with k_i8 in that [b,lk,h,d] layout. */
int tdb200_sla_kmean_partial(const void* k, int dtype, int64_t b, int64_t l, int64_t h, int64_t d, float* partial, void* stream);
int tdb200_sla_kmean_final(const float* partial, int64_t b, int64_t h, int64_t chunks, int64_t d, int64_t l_total, float* kmean,
                           void* stream);
int tdb200_sla_quant_k_seq(const void* k, const float* kmean, int dtype, int64_t b, int64_t l, int64_t h, int64_t d,
                           int8_t* k_i8, float* k_scale, void* k_pool, void* stream);
int tdb200_sla_attn_fwd_kseq(const int8_t* q_i8, const float* q_scale, const int8_t* k_i8, const float* k_scale,
                             const void* v, const void* q, int dtype, const int32_t* lut, int64_t topk, const void* kvw,
                             const float* ksum, const float* proj_b, void* out, int64_t b, int64_t l, int64_t lk,
                             int64_t h, int64_t d, float sm_scale, void* stream);
/* The non-quantised SLA path (reference: Triton _attn_fwd, turbodiffusion/SLA/kernel.py:33-82, used by SparseLinearAttention
 * when --attention_type sla): the same fused kernel with Q.K^T as a 16-bit tensor-core product on the un-quantised q, k
 * [b,l,h,d] (fp32 scores, exp2 softmax, P rounded to T before P.V, :60-73); no q/k scales, no key smoothing. */
int tdb200_sla_attn_fwd_qk16(const void* q, const void* k, const void* v, int dtype, const int32_t* lut, int64_t topk,
                             const void* kvw, const float* ksum, const float* proj_b, void* out, int64_t b, int64_t l,
                             int64_t lk, int64_t h, int64_t d, float sm_scale, void* stream);
/* Second-generation fused kernel (persistent tiles, two softmax threads per query row, linear branch folded into the
 * P.V accumulator); same arguments plus `feature`: 0 softmax, 1 elu+1, 2 relu feature map of the linear branch
 * (SLA/core.py:57-73; the moments must have been built with the same map). */
int tdb200_sla_attn_fwd_v2(const int8_t* q_i8, const float* q_scale, const int8_t* k_i8, const float* k_scale,
                           const void* v, const void* q, int dtype, const int32_t* lut, int64_t topk, const void* kvw,
                           const float* ksum, const float* proj_b, void* out, int64_t b, int64_t l, int64_t lk,
                           int64_t h, int64_t d, float sm_scale, int feature, void* stream);

/* ---------------------------------------------------------------------------------------------
 * a12. LTX-2 (TurboT2AV) prologue variants   (ltx_core/model/transformer/transformer.py:21-94; Triton fast path
 *      ltx_distillation/fast_norm_kernels.py:388-473).  x, y, residual [b, tokens, n] 16-bit; table [num_ada, n] fp32;
 *      timestep [b, ts_tokens, num_ada*n] 16-bit with ts_tokens in {1, tokens}; ada value i = table[i] + timestep[.., i, :].
 *      fp32 math, one rounding to the io dtype.
 *   modulated_rms_norm_ada:  y = rms_norm(x, eps) * (1 + ada[scale_index]) + ada[shift_index]
 *   modulate_ada:            y = x * (1 + ada[scale_index]) + ada[shift_index]
 *   gated_residual_ada:      y = x + residual * ada[gate_index]
 *   split_rope:              x [b,t,h,d], cos/sin [b,h,t,d/2]:  y[:d/2] = x1*cos - x2*sin,  y[d/2:] = x2*cos + x1*sin
 *                            (ltx_core/model/transformer/rope.py:42-60)
 * ------------------------------------------------------------------------------------------- */
int tdb200_ltx_modulated_rms_norm_ada(const void* x, int dtype, const float* table, const void* timestep, int scale_index,
                                      int shift_index, int num_ada, void* y, int64_t b, int64_t tokens, int64_t ts_tokens,
                                      int64_t n, float eps, void* stream);
int tdb200_ltx_modulate_ada(const void* x, int dtype, const float* table, const void* timestep, int scale_index,
                            int shift_index, int num_ada, void* y, int64_t b, int64_t tokens, int64_t ts_tokens, int64_t n,
                            void* stream);
int tdb200_ltx_gated_residual_ada(const void* x, const void* residual, int dtype, const float* table, const void* timestep,
                                  int gate_index, int num_ada, void* y, int64_t b, int64_t tokens, int64_t ts_tokens,
                                  int64_t n, void* stream);
int tdb200_ltx_split_rope(const void* x, const void* cos_freqs, const void* sin_freqs, int dtype, void* y, int64_t b,
                          int64_t t, int64_t h, int64_t d, void* stream);

/* LTX-2 W8A8 with per-row post-scale (ltx_distillation/tilelang_w8a8.py:16-36, 78-117):
 *   quant_int8_rowwise: x [m,k] 16-bit -> q int8 [m,k], s [m] fp32; scale = max(amax,1e-4)/127, round half away, clip.
 *                       (IEEE division here; the reference's Triton `/` is div.full.f32, so exact .5 ties may differ)
 *   gemm_w8a8_rowwise:  c[i,j] = T( fma( float(sum_k a_q[i,k]*b_q[j,k]) * a_s[i], b_s[j], bias[j] ) ) -- the arithmetic the
 *                       reference's TileLang epilogue executes (I2FP, FMUL, FFMA under nvcc's default -fmad; see
 *                       tools/tilelang_epilogue_probe.py); int32 accumulation over all of K in TMEM, one epilogue per
 *                       tile (no per-K-block dequant).  bias may be NULL (= 0).  k % 128 == 0, n % 8 == 0. */
int tdb200_quant_int8_rowwise(const void* x, int dtype, int64_t m, int64_t k, int8_t* q, float* s, void* stream);
int tdb200_gemm_w8a8_rowwise(const int8_t* a_q, const float* a_s, const int8_t* b_q, const float* b_s, const void* bias,
                             void* c, int c_dtype, int64_t m, int64_t n, int64_t k, void* stream);

/* Diagnostics: runs a 128x128x64 bf16 tcgen05 MMA with a K-major A and an MN-major B tile staged by TMA and
 * writes the fp32 product to d_out [128,128].  a [128,64] bf16 row-major, b [64,128] bf16 row-major (d = a.b). */
int tdb200_selftest_umma_bf16(const void* a, const void* b, float* d_out, void* stream);
/* Diagnostics: phase trace of the fused attention kernel.  trace (device, 2*64*8 int64) or NULL to disable; see
 * sla_attn.cu (g_attn_trace) for the layout.  Synchronises the device (cudaMemcpyToSymbol). */
int tdb200_debug_set_attn_trace(long long* trace_or_null);
/* Diagnostics: TMEM->register read throughput.  One CTA per SM, `warps` (4/8/12/16) warps each issuing `iters`
 * tcgen05.ld.32x32b.x64 (8 KB per warp instruction), optionally followed by the GEMM's int->float + FMA dequant.
 * cycles_per_cta [#SMs] receives clock64() deltas. */
int tdb200_selftest_tmem_read(int warps, int iters, int convert, long long* cycles_per_cta, float* sink, void* stream);
/* XU (MUFU) throughput probe: mode 0/1/2 = ex2 f32 / bf16x2 / f16x2, 3/4/5 = tanh f32 / bf16x2 / f16x2; one CTA per SM with
 * `warps` warps, 8 independent chains x `iters` per thread; cycles_per_cta[sm_count]. Diagnostics only. */
int tdb200_selftest_mufu(int mode, int warps, int iters, long long* cycles_per_cta, float* sink, void* stream);
/* diagnostics: the exponential pass of the fused attention's softmax warps on register data (variants drop the packing / the row sums) */
int tdb200_selftest_softmax_exps(int variant, int warps, int iters, long long* cycles_per_cta, float* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TDB200_H_ */
