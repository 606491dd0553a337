// a10 (first half). Linear-attention moments of the keys (reference: turbodiffusion/SLA/core.py:243-247):
//   phi = softmax over the head dim (rounded to the 16-bit type),
//   kv[b,h,dv,dk] += sum_l v[l,dv] * phi(k)[l,dk]        (stored transposed: rows = value channel, cols = key channel)
//   ksum[b,h,dk]  += sum_l phi(k)[l,dk]
// Both outputs are ACCUMULATED (caller zeroes them), so sequence shards combine by plain addition (one all-reduce across
// GPUs).  The L axis of one head is split over `splits` CTAs.  tdb200_sla_linear_moments_ws combines the split partials in a
// fixed order: every CTA stores its partial to a workspace slot, then a second kernel sums the slots in ascending split order
// and adds the sum once (bit-reproducible).  The workspace entry points fix `splits` from the shape alone (kSplitTarget), so
// the result does not depend on the SM count either.  The older entry points add the partials with fp32 red.global.add in
// arrival order instead (the last bits of kv / ksum then vary from run to run).
// A second kernel rather than a last-CTA-reduces ticket: no counter state that must be zero before the call, and the
// ~0.8 MB of partials per head at shape A are summed by the whole GPU instead of by one SM at the tail of the kernel.
//
// CTA = 6 warps, 128 key rows per tile.  warps 0-3: thread == key row: load the row, softmax over D (MUFU ex2), write
// phi(k) into shared memory in the MN-major 128B-swizzled operand layout, then column-sum the tile for ksum.
// warp 4: TMA loads of the V tile (consumed MN-major as the A operand: M = value channel).  warp 5: tcgen05.mma
// kind::f16, D[128(dv) x 128(dk)] += V^T . phi(K), fp32 accumulator in TMEM across all tiles of this CTA.
// 64-wide heads (SLA/core.py:207) run through the same 128x128 tile as PAIRS of adjacent heads: in the [L, H, 64] layout two
// heads are 128 contiguous columns, i.e. exactly one 128-wide row of V and of K.  The tensor core then produces
// [V_a | V_b]^T . [phi(K_a) | phi(K_b)]; its two diagonal 64x64 blocks are the two heads' moment matrices (the off-diagonal
// blocks are discarded), so a pair costs what one 128-wide head costs.  phi is evaluated per 64-wide half.
// Feature maps (SLA/core.py:57-73): 0 softmax over the head dim, 1 elu(x)+1, 2 relu(x).
#include <type_traits>

#include "common.cuh"
#include "host_common.h"

namespace {
using namespace tdb;

constexpr int D = 128;
constexpr int kRowsPerTile = 128;
constexpr int kThreads = 192;
constexpr uint32_t kOperandBytes = kRowsPerTile * D * 2;  // 32 KB: two 64-channel blocks of 128 rows x 128 B
constexpr uint32_t kBlockBytes = kOperandBytes / 2;       // 16 KB
constexpr uint32_t kOffV = 0;                             // 2 stages
constexpr uint32_t kOffPhi = 2 * kOperandBytes;           // 2 stages
constexpr uint32_t kOffBars = 4 * kOperandBytes;          // 128 KB
constexpr size_t kSmemBytes = 1024 + kOffBars + 128;
constexpr float kLog2e = 1.4426950408889634f;

enum Bar { kVFull = 0 /*2*/, kPhiFull = 2 /*2*/, kStageEmpty = 4 /*2*/, kAccFull = 6, kNumBars = 7 };

struct MomParams {
  const void* k;
  float* kv;
  float* ksum;
  float* part;   // NULL: red.global.add into kv / ksum; else split s stores its partial to part + s * slot (plain stores)
  int64_t slot;  // floats per workspace slot: kv [b,h,hd,hd] at offset 0, then ksum [b,h,hd] at offset kv_elems
  int64_t kv_elems;
  int l, h, tiles, splits;
  int hd;        // 128, or 64 (two heads per 128-wide row; `h` is then the number of REAL heads, grid.x = ceil(h/2) pairs)
  int feature;   // 0 softmax, 1 elu+1, 2 relu
};

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// accumulate into kv / ksum (atomic) or store into this CTA's own workspace slot (plain)
__device__ __forceinline__ void put_v4(bool plain, float* addr, const uint32_t* o) {
  if (plain)
    *reinterpret_cast<float4*>(addr) = make_float4(__uint_as_float(o[0]), __uint_as_float(o[1]), __uint_as_float(o[2]),
                                                   __uint_as_float(o[3]));
  else
    red_add_v4(addr, __uint_as_float(o[0]), __uint_as_float(o[1]), __uint_as_float(o[2]), __uint_as_float(o[3]));
}
__device__ __forceinline__ void put_f32(bool plain, float* addr, float x) {
  if (plain) *addr = x;
  else atomicAdd(addr, x);
}

template <typename T, bool kPair>
__global__ void __launch_bounds__(kThreads, 1)
sla_moments_kernel(const __grid_constant__ CUtensorMap tmap_v, MomParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // 1024-aligned, stays a shared-space pointer
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int hh = blockIdx.x, split = blockIdx.y, b = blockIdx.z;  // heads (or head pairs) fastest: DRAM page locality of [L, H, D]
  constexpr bool pair = kPair;
  const int head0 = pair ? 2 * hh : hh;                            // first real head of this CTA
  const bool second_ok = !pair || head0 + 1 < p.h;                 // odd head count: the last pair has one real head
  const int64_t row_elems = int64_t(p.h) * p.hd;                   // elements per token row of k / v
  const int my_tiles = (p.tiles - split + p.splits - 1) / p.splits;  // tiles split, split+splits, ...
  const bool plain = p.part != nullptr;
  float* const kv_out = plain ? p.part + split * p.slot : p.kv;
  float* const ksum_out = plain ? p.part + split * p.slot + p.kv_elems : p.ksum;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars[kVFull + i], 1);
      mbar_init(&bars[kPhiFull + i], 4);
      mbar_init(&bars[kStageEmpty + i], 1);
    }
    mbar_init(&bars[kAccFull], 1);
    mbar_fence_init();
  }
  if (warp == 5) tmem_alloc<128>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  if (my_tiles <= 0) {  // nothing to do (more splits than tiles; the host clamps splits <= tiles); still release TMEM
    __syncthreads();
    if (warp == 5) tmem_dealloc<128>(tmem_base);
    return;
  }

  if (warp == 4) {
    if (lane == 0) {
      tma_prefetch_desc(&tmap_v);
      for (int i = 0; i < my_tiles; ++i) {
        const int st = i & 1, tile = split + i * p.splits;
        mbar_wait(&bars[kStageEmpty + st], ((i >> 1) & 1) ^ 1);
        mbar_expect_tx(&bars[kVFull + st], kOperandBytes);
        uint8_t* sv = smem + kOffV + st * kOperandBytes;
        // 128-wide head: columns [0,64) and [64,128) of head hh; 64-wide heads: heads 2hh and 2hh+1 (a missing second
        // head is out of range in the head dimension, which TMA fills with zeros)
        tma_load_4d(sv, &tmap_v, &bars[kVFull + st], 0, head0, tile * kRowsPerTile, b);
        tma_load_4d(sv + kBlockBytes, &tmap_v, &bars[kVFull + st], pair ? 0 : 64, pair ? head0 + 1 : head0, tile * kRowsPerTile, b);
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      constexpr bool is_bf16 = std::is_same<T, __nv_bfloat16>::value;
      constexpr uint32_t idesc = make_idesc(kDFmtF32, is_bf16 ? kFmtBF16 : kFmtF16, is_bf16 ? kFmtBF16 : kFmtF16, 1, 1, D, D);
      const uint32_t sbase = smem_u32(smem);
      for (int i = 0; i < my_tiles; ++i) {
        const int st = i & 1;
        mbar_wait(&bars[kVFull + st], (i >> 1) & 1);
        mbar_wait(&bars[kPhiFull + st], (i >> 1) & 1);
        tc_fence_after_sync();
        const uint64_t adesc = make_desc_mnmajor_sw128(sbase + kOffV + st * kOperandBytes, kBlockBytes);
        const uint64_t bdesc = make_desc_mnmajor_sw128(sbase + kOffPhi + st * kOperandBytes, kBlockBytes);
#pragma unroll
        for (int ks = 0; ks < kRowsPerTile / 16; ++ks)  // K = 16 key rows per MMA: +2048 B in both operands
          umma_f16_ss(tmem_base, adesc + uint64_t(ks * 128), bdesc + uint64_t(ks * 128), idesc, (i > 0 || ks > 0) ? 1u : 0u);
        umma_commit(&bars[kStageEmpty + st]);
      }
      umma_commit(&bars[kAccFull]);
    }
  } else {
    const int r = warp * 32 + lane;  // key row inside the tile; later: value channel (TMEM lane) / key channel (ksum)
    float ksum_acc = 0.f;
    // The key rows of tile i+1 are requested before tile i is transformed (16 independent 16-byte loads per thread in flight
    // under the exponentials), and phi needs ONE exponential per element: e_j is kept in fp32 registers until the row sum is
    // known.  (Round 1 loaded, waited, and evaluated every exponential twice: 9.8k clk per 128-row tile.)
    auto load_row = [&](int i, uint4 (&dst)[D / 8]) {
      const int64_t row = int64_t(split + i * p.splits) * kRowsPerTile + r;
      const int nload = (i < my_tiles && row < p.l) ? (second_ok ? D / 8 : D / 16) : 0;   // missing second head: zeros
      const uint4* src = reinterpret_cast<const uint4*>(static_cast<const T*>(p.k) +
                                                        (int64_t(b) * p.l + (row < p.l ? row : 0)) * row_elems + int64_t(head0) * p.hd);
#pragma unroll
      for (int c = 0; c < D / 8; ++c) {
        dst[c] = make_uint4(0u, 0u, 0u, 0u);
        if (c < nload) dst[c] = ldg_nc_v4(src + c);
      }
    };
    uint4 cur[D / 8];
    load_row(0, cur);
    for (int i = 0; i < my_tiles; ++i) {
      const int st = i & 1, tile = split + i * p.splits;
      const int64_t row = int64_t(tile) * kRowsPerTile + r;
      uint4 nxt[D / 8];
      load_row(i + 1, nxt);
      uint32_t w[D / 2];
#pragma unroll
      for (int c = 0; c < D / 8; ++c) { w[4 * c] = cur[c].x; w[4 * c + 1] = cur[c].y; w[4 * c + 2] = cur[c].z; w[4 * c + 3] = cur[c].w; }
      if (row < p.l) {
        // phi over each segment of the row (one 128-wide segment, or two 64-wide segments for a pair of 64-wide heads)
        constexpr int kSeg = kPair ? 2 : 1, kWps = (D / 2) / kSeg;   // segments, 32-bit words per segment
#pragma unroll
        for (int sgm = 0; sgm < kSeg; ++sgm) {
          const int w0 = sgm * kWps;
          if (p.feature == 0) {
            float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
            for (int q = 0; q < kWps; q += 2) {
              m0 = fmaxf(m0, fmaxf(F16Traits<T>::lo(w[w0 + q]), F16Traits<T>::hi(w[w0 + q])));
              m1 = fmaxf(m1, fmaxf(F16Traits<T>::lo(w[w0 + q + 1]), F16Traits<T>::hi(w[w0 + q + 1])));
            }
            const float off = fmaxf(m0, m1) * kLog2e;
            float e[2 * kWps];
            float sa = 0.f, sb = 0.f, sc4 = 0.f, sd = 0.f;  // independent chains
#pragma unroll
            for (int q = 0; q < kWps; q += 2) {
              e[2 * q] = fast_exp2(fmaf(F16Traits<T>::lo(w[w0 + q]), kLog2e, -off));
              e[2 * q + 1] = fast_exp2(fmaf(F16Traits<T>::hi(w[w0 + q]), kLog2e, -off));
              e[2 * q + 2] = fast_exp2(fmaf(F16Traits<T>::lo(w[w0 + q + 1]), kLog2e, -off));
              e[2 * q + 3] = fast_exp2(fmaf(F16Traits<T>::hi(w[w0 + q + 1]), kLog2e, -off));
              sa += e[2 * q]; sb += e[2 * q + 1]; sc4 += e[2 * q + 2]; sd += e[2 * q + 3];
            }
            const float inv = 1.0f / ((sa + sb) + (sc4 + sd));
#pragma unroll
            for (int q = 0; q < kWps; ++q) w[w0 + q] = F16Traits<T>::pack(e[2 * q] * inv, e[2 * q + 1] * inv);
          } else {
#pragma unroll
            for (int q = 0; q < kWps; ++q) {
              const float a = F16Traits<T>::lo(w[w0 + q]), c = F16Traits<T>::hi(w[w0 + q]);
              const float fa = p.feature == 1 ? (a > 0.f ? a + 1.0f : fast_exp2(a * kLog2e)) : fmaxf(a, 0.f);
              const float fc = p.feature == 1 ? (c > 0.f ? c + 1.0f : fast_exp2(c * kLog2e)) : fmaxf(c, 0.f);
              w[w0 + q] = F16Traits<T>::pack(fa, fc);
            }
          }
        }
        if (!second_ok) {
#pragma unroll
          for (int q = D / 4; q < D / 2; ++q) w[q] = 0u;
        }
      } else {
#pragma unroll
        for (int q = 0; q < D / 2; ++q) w[q] = 0u;
      }
#pragma unroll
      for (int c = 0; c < D / 8; ++c) cur[c] = nxt[c];
      // stage free? (the MMA that read it two tiles ago has retired)
      mbar_wait(&bars[kStageEmpty + st], ((i >> 1) & 1) ^ 1);
      uint8_t* sphi = smem + kOffPhi + st * kOperandBytes;
#pragma unroll
      for (int c = 0; c < 16; ++c)
        *reinterpret_cast<uint4*>(sphi + (c >> 3) * kBlockBytes + r * 128 + (((c & 7) ^ (r & 7)) << 4)) =
            make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
      fence_proxy_async_smem();
      named_bar_sync(1, 128);  // all 128 rows of the tile are written (also orders the ksum reads below)
      if (lane == 0) mbar_arrive(&bars[kPhiFull + st]);
      // ---- ksum: thread r sums key channel r over the 128 rows of the tile
      {
        const uint8_t* colbase = sphi + (r >> 6) * kBlockBytes + (r & 7) * 2;
        const int chunk = (r & 63) >> 3;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
        for (int rr = 0; rr < kRowsPerTile; rr += 4) {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const unsigned short raw =
                *reinterpret_cast<const unsigned short*>(colbase + (rr + u) * 128 + ((chunk ^ ((rr + u) & 7)) << 4));
            s4[u] += F16Traits<T>::lo(static_cast<uint32_t>(raw));
          }
        }
        ksum_acc += (s4[0] + s4[1]) + (s4[2] + s4[3]);
      }
    }
    // thread r holds key channel r of the 128-wide row: head0's channel r, or (pairs) channel r-64 of head0+1
    if (!pair) {
      put_f32(plain, ksum_out + (int64_t(b) * p.h + head0) * D + r, ksum_acc);
    } else if (r < 64 || second_ok) {
      put_f32(plain, ksum_out + (int64_t(b) * p.h + head0 + (r >> 6)) * 64 + (r & 63), ksum_acc);
    }
    // ---- kv: TMEM lane r = value channel r, 128 key channels
    mbar_wait(&bars[kAccFull], 0);
    tc_fence_after_sync();
    if (!pair) {
      float* dst = kv_out + ((int64_t(b) * p.h + head0) * D + r) * D;
#pragma unroll
      for (int c = 0; c < D / 32; ++c) {
        uint32_t o[32];
        tmem_ld_x32(tmem_base + (uint32_t(warp * 32) << 16) + c * 32, o);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 32; q += 4) put_v4(plain, dst + c * 32 + q, o + q);
      }
    } else {
      // lane r = value channel (r & 63) of head0 + (r >> 6); its diagonal block is key columns [64*(r>>6), +64)
      const int sub = r >> 6;                        // warp-uniform (warps 0,1 -> head0; warps 2,3 -> head0+1)
      float* dst = kv_out + ((int64_t(b) * p.h + head0 + sub) * 64 + (r & 63)) * 64;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t o[32];
        tmem_ld_x32(tmem_base + (uint32_t(warp * 32) << 16) + sub * 64 + c * 32, o);
        tmem_ld_wait();
        if (sub == 0 || second_ok) {
#pragma unroll
          for (int q = 0; q < 32; q += 4) put_v4(plain, dst + c * 32 + q, o + q);
        }
      }
    }
    tc_fence_before_sync();
  }
  __syncthreads();
  if (warp == 5) {
    tc_fence_after_sync();
    tmem_dealloc<128>(tmem_base);
  }
}

// kv += sum_s part[s][0, kv_elems), ksum += sum_s part[s][kv_elems, slot): one float4 per thread, splits summed in
// ascending order in fp32, then added to the accumulator once.
__global__ void __launch_bounds__(256) moments_reduce_kernel(const float4* __restrict__ part, float4* kv, float4* ksum,
                                                              int64_t kv4, int64_t slot4, int splits) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= slot4) return;
  float4 acc = part[i];
  for (int s = 1; s < splits; ++s) {
    const float4 x = part[s * slot4 + i];
    acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
  }
  float4* dst = i < kv4 ? kv + i : ksum + (i - kv4);
  float4 y = *dst;
  y.x += acc.x; y.y += acc.y; y.z += acc.z; y.w += acc.w;
  *dst = y;
}

// CTAs per head unit for the workspace entry points: one wave of a 148-SM B200 at b * units <= 148, a function of the shape
// only (the workspace size is then known without a device, and the summation order is the same on every GPU).
constexpr int kSplitTarget = 148;

int64_t units_of(int64_t h, int64_t d) { return d == 128 ? h : cdiv64(h, 2); }  // CTAs along x: heads, or pairs of 64-wide heads

int splits_of(int64_t sms, int64_t b, int64_t l, int64_t h, int64_t d) {
  const int64_t tiles = cdiv64(l, kRowsPerTile);
  int64_t splits = sms / (b * units_of(h, d));
  if (splits < 1) splits = 1;
  if (splits > tiles) splits = tiles;
  return int(splits);
}

int check_shape(const void* k, const void* v, int64_t b, int64_t l, int64_t h, int64_t d, int feature, float* kv, float* ksum) {
  if (!k || !v || !kv || !ksum) return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments: null pointer");
  if (b <= 0 || l <= 0 || h <= 0 || l > 0x7FFFFFFF) return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments: bad shape");
  if (d != 64 && d != 128) return fail(TDB200_ERR_UNSUPPORTED, "sla_linear_moments: head dim %lld (64 or 128, SLA/core.py:207)", (long long)d);
  if (feature < 0 || feature > 2) return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments: feature map tag %d", feature);
  if (h > 65535 || b > 65535) return fail(TDB200_ERR_UNSUPPORTED, "sla_linear_moments: h or b too large");
  if (!aligned16(k) || !aligned16(kv)) return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments: buffers must be 16-byte aligned");
  return TDB200_OK;
}

}  // namespace

// part == NULL: the split partials are added into kv / ksum with fp32 atomics (order of arrival).  Otherwise part holds
// `splits` slots of MomParams::slot floats and a second kernel reduces them in a fixed order.
static int moments_impl(const void* k, const void* v, int dtype, int64_t b, int64_t l, int64_t h, int64_t d, int feature,
                        float* kv, float* ksum, float* part, int splits, void* stream) {
  using namespace tdb;
  if (int rc = require_sm100()) return rc;
  const CUtensorMapDataType t16 = dtype == TDB200_DTYPE_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUtensorMap tv;
  {
    const uint64_t dims[4] = {uint64_t(d), uint64_t(h), uint64_t(l), uint64_t(b)};
    const uint64_t str[3] = {uint64_t(d * 2), uint64_t(h * d * 2), uint64_t(l * h * d * 2)};
    const uint32_t box[4] = {64, 1, kRowsPerTile, 1};
    if (int rc = make_tmap_4d(&tv, v, t16, 2, dims, str, box)) return rc;
  }
  MomParams p;
  p.k = k;
  p.kv = kv;
  p.ksum = ksum;
  p.part = part;
  p.kv_elems = b * h * d * d;
  p.slot = p.kv_elems + b * h * d;
  p.l = int(l);
  p.h = int(h);
  p.hd = int(d);
  p.feature = feature;
  p.tiles = int(cdiv64(l, kRowsPerTile));
  p.splits = splits;
  dim3 grid(static_cast<unsigned>(units_of(h, d)), splits, static_cast<unsigned>(b));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = TDB200_OK;
#define TDB_MOM2(T, PAIR)                                                                                          \
  do {                                                                                                              \
    static bool attr_done[64] = {false};                                                                            \
    if (int e = set_max_dynamic_smem_once(reinterpret_cast<const void*>(sla_moments_kernel<T, PAIR>), kSmemBytes, attr_done, \
                                          "cudaFuncSetAttribute(sla_moments)"))                                    \
      return e;                                                                                                     \
    sla_moments_kernel<T, PAIR><<<grid, kThreads, kSmemBytes, st>>>(tv, p);                                         \
    rc = check_launch("sla_moments_kernel");                                                                        \
  } while (0)
#define TDB_MOM(T) do { if (d == 64) { TDB_MOM2(T, true); } else { TDB_MOM2(T, false); } } while (0)
  if (dtype == TDB200_DTYPE_BF16) TDB_MOM(__nv_bfloat16);
  else if (dtype == TDB200_DTYPE_FP16) TDB_MOM(__half);
  else return fail(TDB200_ERR_UNSUPPORTED, "sla_linear_moments: dtype tag %d", dtype);
#undef TDB_MOM2
#undef TDB_MOM
  if (rc != TDB200_OK || part == nullptr) return rc;
  const int64_t slot4 = p.slot / 4;   // kv_elems and slot are multiples of 4 (d * d and d are)
  moments_reduce_kernel<<<static_cast<unsigned>(cdiv64(slot4, 256)), 256, 0, st>>>(
      reinterpret_cast<const float4*>(part), reinterpret_cast<float4*>(kv), reinterpret_cast<float4*>(ksum), p.kv_elems / 4,
      slot4, splits);
  return check_launch("moments_reduce_kernel");
}

extern "C" int tdb200_sla_linear_moments(const void* k, const void* v, int dtype, int64_t b, int64_t l, int64_t h,
                                         int64_t d, float* kv, float* ksum, void* stream) {
  return tdb200_sla_linear_moments_ex(k, v, dtype, b, l, h, d, 0, kv, ksum, stream);
}

extern "C" int tdb200_sla_linear_moments_ex(const void* k, const void* v, int dtype, int64_t b, int64_t l, int64_t h,
                                            int64_t d, int feature, float* kv, float* ksum, void* stream) {
  if (int rc = check_shape(k, v, b, l, h, d, feature, kv, ksum)) return rc;
  return moments_impl(k, v, dtype, b, l, h, d, feature, kv, ksum, nullptr, splits_of(tdb::sm_count(), b, l, h, d), stream);
}

extern "C" int tdb200_sla_linear_moments_workspace(int64_t b, int64_t l, int64_t h, int64_t d, int64_t* bytes) {
  using namespace tdb;
  if (!bytes) return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments_workspace: null pointer");
  if (b <= 0 || l <= 0 || h <= 0 || l > 0x7FFFFFFF || h > 65535 || b > 65535)
    return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments_workspace: bad shape");
  if (d != 64 && d != 128) return fail(TDB200_ERR_UNSUPPORTED, "sla_linear_moments_workspace: head dim %lld (64 or 128)", (long long)d);
  *bytes = int64_t(splits_of(kSplitTarget, b, l, h, d)) * (b * h * d * (d + 1)) * int64_t(sizeof(float));
  return TDB200_OK;
}

extern "C" int tdb200_sla_linear_moments_ws(const void* k, const void* v, int dtype, int64_t b, int64_t l, int64_t h,
                                            int64_t d, int feature, float* kv, float* ksum, void* workspace,
                                            int64_t workspace_bytes, void* stream) {
  using namespace tdb;
  if (int rc = check_shape(k, v, b, l, h, d, feature, kv, ksum)) return rc;
  if (!workspace) return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments_ws: null workspace");
  if (!aligned16(ksum) || !aligned16(workspace))
    return fail(TDB200_ERR_INVALID_ARG, "sla_linear_moments_ws: ksum and workspace must be 16-byte aligned");
  int64_t need = 0;
  if (int rc = tdb200_sla_linear_moments_workspace(b, l, h, d, &need)) return rc;
  if (workspace_bytes < need)
    return fail(TDB200_ERR_WORKSPACE, "sla_linear_moments_ws: workspace of %lld bytes, %lld needed", (long long)workspace_bytes,
                (long long)need);
  return moments_impl(k, v, dtype, b, l, h, d, feature, kv, ksum, static_cast<float*>(workspace),
                      splits_of(kSplitTarget, b, l, h, d), stream);
}

// ---- kvw = T(proj_w . kv): the linear branch's output projection folded into the moment matrix (SLA/core.py:243-253:
// proj_l(phi(q) kv / den) == phi(q) (proj_w kv)^T / den + b), one launch instead of a library sgemm plus casts.
//   proj_w [d_out, d_v] fp32, kv [bh, d_v, d_k] fp32  ->  kvw [bh, d_out, d_k] T;  fp32 FMA chain over d_v in ascending order.
namespace {
template <typename T, int D>
__global__ void __launch_bounds__(D) project_moments_kernel(const float* __restrict__ w, const float* __restrict__ kv,
                                                            T* __restrict__ out) {
  constexpr int kRows = 32;                      // output rows (d_out) per CTA
  __shared__ float ws[kRows][D];
  const int bh = blockIdx.x, o0 = blockIdx.y * kRows, k = threadIdx.x;
  for (int i = threadIdx.x; i < kRows * D; i += D) ws[i / D][i % D] = __ldg(w + int64_t(o0 + i / D) * D + (i % D));
  __syncthreads();
  float acc[kRows];
#pragma unroll
  for (int i = 0; i < kRows; ++i) acc[i] = 0.f;
  const float* kvp = kv + int64_t(bh) * D * D + k;
#pragma unroll 4
  for (int v = 0; v < D; ++v) {
    const float x = __ldg(kvp + int64_t(v) * D);
#pragma unroll
    for (int i = 0; i < kRows; ++i) acc[i] = fmaf(ws[i][v], x, acc[i]);
  }
  T* op = out + (int64_t(bh) * D + o0) * D + k;
#pragma unroll
  for (int i = 0; i < kRows; ++i) op[int64_t(i) * D] = static_cast<T>(acc[i]);
}
}  // namespace

extern "C" int tdb200_sla_project_moments(const float* proj_w, const float* kv, int dtype, int64_t bh, int64_t d, void* kvw,
                                          void* stream) {
  using namespace tdb;
  if (!proj_w || !kv || !kvw) return fail(TDB200_ERR_INVALID_ARG, "sla_project_moments: null pointer");
  if (bh <= 0 || bh > 0x7FFFFFFF) return fail(TDB200_ERR_INVALID_ARG, "sla_project_moments: bad shape");
  if (d != 64 && d != 128) return fail(TDB200_ERR_UNSUPPORTED, "sla_project_moments: head dim %lld (64 or 128)", (long long)d);
  if (int rc = require_sm100()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid(static_cast<unsigned>(bh), static_cast<unsigned>(d / 32));
#define TDB_PM(T, D) project_moments_kernel<T, D><<<grid, D, 0, st>>>(proj_w, kv, static_cast<T*>(kvw)); return check_launch("project_moments_kernel")
  if (dtype == TDB200_DTYPE_BF16) {
    if (d == 128) { TDB_PM(__nv_bfloat16, 128); }
    TDB_PM(__nv_bfloat16, 64);
  }
  if (dtype == TDB200_DTYPE_FP16) {
    if (d == 128) { TDB_PM(__half, 128); }
    TDB_PM(__half, 64);
  }
#undef TDB_PM
  return fail(TDB200_ERR_UNSUPPORTED, "sla_project_moments: dtype tag %d", dtype);
}
