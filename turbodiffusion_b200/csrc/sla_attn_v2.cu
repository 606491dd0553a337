// a9 + a10 (second generation).  Fused SageSLA attention forward as a PERSISTENT kernel: two CTAs per SM walk the
// (query block, head, batch) tiles; per tile
//   block-sparse INT8 Q.K^T -> online softmax (exp2) -> 16-bit P.V accumulated in tensor memory,
//   then the linear branch is folded INTO the same accumulator:  O += (phi(q) * l/den) . KVW^T,   out = O / l + b,
// so one TMEM accumulator, one epilogue read, no second product to merge.
//   reference: Sage call site turbodiffusion/SLA/core.py:231-235 (arithmetic in third-party SpargeAttn, unpinned);
//   the in-tree statement of the same attention is the Triton kernel SLA/kernel.py:33-82 (tail masking :57-62, exp2 with
//   qk_scale*log2e :60, row sum from unrounded P :71, P cast before P.V :73); linear branch + merge SLA/core.py:243-253.
//
// CTA = 10 warps.  warps 0-7: softmax; TWO threads per query row (warp w and w+4 share TMEM lane quarter w%4; thread half
//   hf = w/4 owns key columns [32*hf, 32*hf+32) of every S tile, the matching half of the O columns and of the q row):
//   four warps per scheduler across the two co-resident CTAs instead of two, and half the serial work per iteration.
//   Row maxima / sums are exchanged through shared memory under a 64-thread named barrier per lane quarter.
//   warp 8: TMA producer (K and V rings that run on across tile boundaries, double-buffered Q tile, next tile's LUT).
//   warp 9: MMA issuer.
// Tensor memory (256 columns): S[2] int32 128x64 at columns [0,128) | O fp32 128xHD at [128, 128+HD).
//   P(j) (16-bit, 32 columns) is written over the S buffer it was computed from and P.V reads it from there (.ts form);
//   the in-order tensor pipe keeps Q.K^T(j+2) behind P.V(j).  After a tile's last key block the free S buffer receives
//   the scaled phi(q) rows (HD/2 columns) and one more .ts MMA adds the linear branch to O.
// Shared memory (HD = 128): Q int8 2x16 KB | K int8 3x8 KB | V 16-bit 3x16 KB  = 104 KB + LUT + barriers, two CTAs per SM.
//   KVW (the proj_l-folded moment matrix of the head) travels through the V ring as the tile's last two entries.
// The O accumulator is only rescaled when a row maximum grows by more than 2^8 (lazy rescale): P stays <= 256.
#include <type_traits>

#include "common.cuh"
#include "host_common.h"

namespace {
using namespace tdb;

constexpr int BLKQ = 128, BLKK = 64;
constexpr int kSoftmaxWarps = 8, kTmaWarp = 8, kMmaWarp = 9;
constexpr int kThreads = 320;
constexpr int kStages = 3;
constexpr uint32_t kTmemCols = 256;
constexpr uint32_t kColS = 0, kColO = 128;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kRescaleThreshold = 8.0f;  // log2 domain

template <int HD>
struct Cfg {
  static constexpr uint32_t kQBytes = BLKQ * HD;            // int8
  static constexpr uint32_t kKBytes = BLKK * HD;            // int8
  static constexpr uint32_t kVBytes = BLKK * HD * 2;        // 16-bit; HD/64 boxes of [64 keys x 128 B]
  static constexpr uint32_t kVBox = BLKK * 128;             // one 64-column box
  static constexpr uint32_t kOffQ = 0;                      // [2]
  static constexpr uint32_t kOffK = kOffQ + 2 * kQBytes;    // [kStages]
  static constexpr uint32_t kOffV = kOffK + kStages * kKBytes;
  static constexpr uint32_t kOffX = kOffV + kStages * kVBytes;  // exchange area: [2][2][128] floats max, [2][128] x 3 sums
  static constexpr uint32_t kXBytes = (2 * 2 * 128 + 3 * 2 * 128) * 4;
  static constexpr uint32_t kOffBars = kOffX + kXBytes;
  static constexpr uint32_t kBarBytes = 512;
  static constexpr uint32_t kOffLut = kOffBars + kBarBytes;
  static constexpr int kKvwEntries = HD / 64;               // V-ring entries taken by the folded moment matrix
};

struct AttnParams {
  const float* q_scale;   // [b,h,mblk]
  const float* k_scale;   // [b,h,nblk]
  const void* q;          // [b,l,h,d] T (linear branch)
  const int32_t* lut;     // [b,h,mblk,topk]
  const float* ksum;      // [b,h,d]
  const float* proj_b;    // [d]
  void* out;              // [b,l,h,d] T
  int l, lk, h, mblk, nblk, topk, tiles, feature;  // feature: 0 softmax, 1 elu+1, 2 relu (SLA/core.py:57-73)
  float sm_scale;
};

enum Bar {
  kQFull = 0 /*2*/, kQFree = 2 /*2*/, kKFull = 4 /*3*/, kKEmpty = 7 /*3*/, kVFull = 10 /*3*/, kVEmpty = 13 /*3*/,
  kSFull = 16 /*2*/, kPFull = 18, kPvDone = 19, kPhiFull = 20, kOFull = 21, kOFree = 22, kLutFull = 23 /*2*/,
  kLutFree = 25 /*2*/, kNumBars = 27
};

__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// tile id -> (query block, head, batch); heads fastest so concurrently running CTAs read whole [row, H*D] lines of V
__device__ __forceinline__ void tile_coords(int tile, const AttnParams& p, int& m_blk, int& hh, int& b) {
  hh = tile % p.h;
  const int t2 = tile / p.h;
  m_blk = t2 % p.mblk;
  b = t2 / p.mblk;
}

template <typename T>
__device__ __forceinline__ float feat(float x, float off_log2, int feature) {
  // softmax numerator exp(x - max) | elu(x)+1 | relu(x)
  if (feature == 0) return fast_exp2(fmaf(x, kLog2e, -off_log2));
  if (feature == 1) return x > 0.f ? x + 1.0f : fast_exp2(x * kLog2e);
  return fmaxf(x, 0.f);
}

template <typename T, int HD>
__global__ void __launch_bounds__(kThreads, 2)
sla_attn_v2_kernel(const __grid_constant__ CUtensorMap tmap_q8, const __grid_constant__ CUtensorMap tmap_k8,
                   const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_kvw,
                   AttnParams p) {
  using C = Cfg<HD>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // 1024-aligned, stays a shared-space pointer
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kOffBars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);
  const uint32_t lut_stride = (uint32_t(p.topk) * 6u + 15u) & ~15u;   // per buffer: [topk] u16 ids, then [topk] f32 k scales
  float* x_max = reinterpret_cast<float*>(smem + C::kOffX);            // [2 parity][2 half][128 rows]
  float* x_sum = x_max + 2 * 2 * 128;                                  // [3 quantities][2 half][128 rows]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T_blocks = p.topk;
  const int my_tiles = (p.tiles - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x);

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars[kQFull + i], 1);
      mbar_init(&bars[kQFree + i], 1);
      mbar_init(&bars[kSFull + i], 1);
      mbar_init(&bars[kLutFull + i], 1);
      mbar_init(&bars[kLutFree + i], kSoftmaxWarps);
    }
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&bars[kKFull + i], 1);
      mbar_init(&bars[kKEmpty + i], 1);
      mbar_init(&bars[kVFull + i], 1);
      mbar_init(&bars[kVEmpty + i], 1);
    }
    mbar_init(&bars[kPFull], kSoftmaxWarps);
    mbar_init(&bars[kPvDone], 1);
    mbar_init(&bars[kPhiFull], kSoftmaxWarps);
    mbar_init(&bars[kOFull], 1);
    mbar_init(&bars[kOFree], kSoftmaxWarps);
    mbar_fence_init();
  }
  if (warp == kMmaWarp) tmem_alloc<kTmemCols>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kTmaWarp) {
    // =============================================================== TMA producer (+ LUT staging by the whole warp)
    if (lane == 0) {
      tma_prefetch_desc(&tmap_q8);
      tma_prefetch_desc(&tmap_k8);
      tma_prefetch_desc(&tmap_v);
      tma_prefetch_desc(&tmap_kvw);
    }
    auto stage_lut = [&](int n) {  // LUT + key scales of this CTA's n-th tile -> buffer n&1
      const int tile = int(blockIdx.x) + n * int(gridDim.x);
      int m_blk, hh, b;
      tile_coords(tile, p, m_blk, hh, b);
      const int bh = b * p.h + hh;
      uint16_t* s_lut = reinterpret_cast<uint16_t*>(smem + C::kOffLut + (n & 1) * lut_stride);
      float* s_ksc = reinterpret_cast<float*>(smem + C::kOffLut + (n & 1) * lut_stride + ((uint32_t(T_blocks) * 2u + 3u) & ~3u));
      if (n >= 2) mbar_wait(&bars[kLutFree + (n & 1)], ((n >> 1) - 1) & 1);  // softmax warps are done with tile n-2's copy
      const int32_t* lut_row = p.lut + (int64_t(bh) * p.mblk + m_blk) * p.topk;
      const float* ksc_row = p.k_scale + int64_t(bh) * p.nblk;
      for (int i = lane; i < T_blocks; i += 32) {
        const int blk = __ldg(lut_row + i);
        s_lut[i] = static_cast<uint16_t>(blk);
        s_ksc[i] = __ldg(ksc_row + blk);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[kLutFull + (n & 1)]);
    };
    uint32_t kq = 0, vq = 0;
    if (my_tiles > 0) stage_lut(0);
    for (int n = 0; n < my_tiles; ++n) {
      const int tile = int(blockIdx.x) + n * int(gridDim.x);
      int m_blk, hh, b;
      tile_coords(tile, p, m_blk, hh, b);
      const int bh = b * p.h + hh;
      const uint16_t* s_lut = reinterpret_cast<const uint16_t*>(smem + C::kOffLut + (n & 1) * lut_stride);
      if (lane == 0) {
        // Q tile -> buffer n&1 (free once the last Q.K^T of tile n-2 has retired)
        if (n >= 2) mbar_wait(&bars[kQFree + (n & 1)], ((n >> 1) - 1) & 1);
        mbar_expect_tx(&bars[kQFull + (n & 1)], C::kQBytes);
        tma_load_4d(smem + C::kOffQ + (n & 1) * C::kQBytes, &tmap_q8, &bars[kQFull + (n & 1)], 0, m_blk * BLKQ, bh, 0);
        for (int j = 0; j < T_blocks; ++j) {
          const int blk = s_lut[j];
          {
            const uint32_t st = kq % kStages, ph = ((kq / kStages) & 1u) ^ 1u;
            mbar_wait(&bars[kKEmpty + st], ph);
            mbar_expect_tx(&bars[kKFull + st], C::kKBytes);
            tma_load_4d(smem + C::kOffK + st * C::kKBytes, &tmap_k8, &bars[kKFull + st], 0, blk * BLKK, bh, 0);
            ++kq;
          }
          {
            const uint32_t st = vq % kStages, ph = ((vq / kStages) & 1u) ^ 1u;
            mbar_wait(&bars[kVEmpty + st], ph);
            mbar_expect_tx(&bars[kVFull + st], C::kVBytes);
            uint8_t* sv = smem + C::kOffV + st * C::kVBytes;
#pragma unroll
            for (int c = 0; c < HD / 64; ++c)
              tma_load_4d(sv + c * C::kVBox, &tmap_v, &bars[kVFull + st], c * 64, hh, blk * BLKK, b);
            ++vq;
          }
        }
        // KVW: HD/64 more V-ring entries, each one 64-wide d_k chunk of the [d_out, d_k] matrix (HD rows x 128 B)
#pragma unroll
        for (int c = 0; c < C::kKvwEntries; ++c) {
          const uint32_t st = vq % kStages, ph = ((vq / kStages) & 1u) ^ 1u;
          mbar_wait(&bars[kVEmpty + st], ph);
          mbar_expect_tx(&bars[kVFull + st], uint32_t(HD) * 128u);
          tma_load_4d(smem + C::kOffV + st * C::kVBytes, &tmap_kvw, &bars[kVFull + st], c * 64, 0, bh, 0);
          ++vq;
        }
      }
      __syncwarp();
      if (n + 1 < my_tiles) stage_lut(n + 1);
      __syncwarp();
    }
  } else if (warp == kMmaWarp) {
    // =============================================================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc_qk = make_idesc(kDFmtS32, kFmtS8, kFmtS8, 0, 0, BLKQ, BLKK);
      constexpr bool is_bf16 = std::is_same<T, __nv_bfloat16>::value;
      constexpr uint32_t f16 = is_bf16 ? kFmtBF16 : kFmtF16;
      constexpr uint32_t idesc_pv = make_idesc(kDFmtF32, f16, f16, 0, 1, BLKQ, HD);   // B = V, MN-major
      constexpr uint32_t idesc_lin = make_idesc(kDFmtF32, f16, f16, 0, 0, BLKQ, HD);  // B = KVW, K-major
      const uint32_t sbase = smem_u32(smem);
      uint32_t g = 0, kq = 0, vq = 0, pc = 0;   // S-buffer slot counter, ring counters, P publishes consumed

      auto issue_qk = [&](int n, uint32_t slot, bool last_of_tile) {
        const uint32_t st = kq % kStages;
        mbar_wait(&bars[kKFull + st], (kq / kStages) & 1u);
        tc_fence_after_sync();
        // int8 rows are HD bytes: 128-byte swizzle for 128-wide heads, 64-byte swizzle for 64-wide heads
        const uint64_t qdesc = HD == 128 ? make_desc_kmajor_sw128(sbase + C::kOffQ + (n & 1) * C::kQBytes)
                                         : make_desc_kmajor_sw64(sbase + C::kOffQ + (n & 1) * C::kQBytes);
        const uint64_t kdesc = HD == 128 ? make_desc_kmajor_sw128(sbase + C::kOffK + st * C::kKBytes)
                                         : make_desc_kmajor_sw64(sbase + C::kOffK + st * C::kKBytes);
#pragma unroll
        for (int ks = 0; ks < HD / 32; ++ks)
          umma_i8_ss(tmem_base + kColS + (slot & 1u) * BLKK, qdesc + uint64_t(ks * 2), kdesc + uint64_t(ks * 2), idesc_qk,
                     ks > 0 ? 1u : 0u);
        umma_commit(&bars[kSFull + (slot & 1u)]);
        umma_commit(&bars[kKEmpty + st]);
        if (last_of_tile) umma_commit(&bars[kQFree + (n & 1)]);
        ++kq;
      };
      auto issue_pv = [&](uint32_t slot, bool first_of_tile, int n) {
        const uint32_t st = vq % kStages;
        mbar_wait(&bars[kPFull], pc & 1u);
        ++pc;
        mbar_wait(&bars[kVFull + st], (vq / kStages) & 1u);
        if (first_of_tile && n > 0) mbar_wait(&bars[kOFree], (n - 1) & 1);  // the epilogue of tile n-1 has read O
        tc_fence_after_sync();
        const uint64_t vdesc = make_desc_mnmajor_sw128(sbase + C::kOffV + st * C::kVBytes, C::kVBox);
#pragma unroll
        for (int ks = 0; ks < BLKK / 16; ++ks)  // K = 16 keys per MMA: P +8 TMEM columns, V +16 rows (2048 B)
          umma_f16_ts(tmem_base + kColO, tmem_base + kColS + (slot & 1u) * BLKK + uint32_t(ks * 8),
                      vdesc + uint64_t(ks * 128), idesc_pv, (!first_of_tile || ks > 0) ? 1u : 0u);
        umma_commit(&bars[kVEmpty + st]);
        umma_commit(&bars[kPvDone]);
        ++vq;
      };

      for (int n = 0; n < my_tiles; ++n) {
        const uint32_t g0 = g;
        if (n == 0) {
          mbar_wait(&bars[kQFull + 0], 0);
          issue_qk(0, g0, T_blocks == 1);
        }
        for (int j = 1; j < T_blocks; ++j) {
          issue_qk(n, g0 + j, j == T_blocks - 1);
          issue_pv(g0 + j - 1, j == 1, n);
        }
        issue_pv(g0 + T_blocks - 1, T_blocks == 1, n);
        g = g0 + T_blocks + 1;  // slot g0+T is the phi(q) slot of this tile
        if (n + 1 < my_tiles) {  // first Q.K^T of the next tile goes out before this tile's linear step
          mbar_wait(&bars[kQFull + ((n + 1) & 1)], ((n + 1) >> 1) & 1);
          issue_qk(n + 1, g, T_blocks == 1);
        }
        // ---- linear branch: O += A[128 x HD] . KVW^T, A = scaled phi(q) in the S buffer of slot g0+T
        mbar_wait(&bars[kPhiFull], n & 1);
        const uint32_t a_tmem = tmem_base + kColS + ((g0 + T_blocks) & 1u) * BLKK;
#pragma unroll
        for (int c = 0; c < C::kKvwEntries; ++c) {
          const uint32_t st = vq % kStages;
          mbar_wait(&bars[kVFull + st], (vq / kStages) & 1u);
          tc_fence_after_sync();
          const uint64_t bdesc = make_desc_kmajor_sw128(sbase + C::kOffV + st * C::kVBytes);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)  // 64-wide d_k chunk = 4 K-steps of 16: A +8 TMEM columns, B +32 bytes
            umma_f16_ts(tmem_base + kColO, a_tmem + uint32_t(c * 32 + ks * 8), bdesc + uint64_t(ks * 2), idesc_lin, 1u);
          umma_commit(&bars[kVEmpty + st]);
          ++vq;
        }
        umma_commit(&bars[kOFull]);
      }
    }
  } else {
    // =============================================================== softmax / correction / epilogue warps
    const int q4 = warp & 3, hf = warp >> 2;
    const int r = q4 * 32 + lane;                        // query row inside the block == TMEM lane
    const uint32_t lane_addr = uint32_t(q4 * 32) << 16;
    const uint32_t pair_bar = 1 + q4;                    // named barrier of the two warps that share these 32 rows
    constexpr float kMagicF = 12582912.0f;               // 1.5 * 2^23: as_float(0x4B400000 + i) == kMagicF + i for |i| < 2^22
    constexpr int kMagicI = 0x4B400000;
    uint32_t s_par0 = 0, s_par1 = 0;                     // phases consumed on SFull[0], SFull[1]
    uint32_t g = 0, pv_waited = 0, p_pub = 0;            // slot counter; PvDone completions consumed; P tiles published

    for (int n = 0; n < my_tiles; ++n) {
      const int tile = int(blockIdx.x) + n * int(gridDim.x);
      int m_blk, hh, b;
      tile_coords(tile, p, m_blk, hh, b);
      const int bh = b * p.h + hh;
      const uint16_t* s_lut = reinterpret_cast<const uint16_t*>(smem + C::kOffLut + (n & 1) * lut_stride);
      const float* s_ksc = reinterpret_cast<const float*>(smem + C::kOffLut + (n & 1) * lut_stride + ((uint32_t(T_blocks) * 2u + 3u) & ~3u));
      const float qsc = __ldg(p.q_scale + int64_t(bh) * p.mblk + m_blk) * p.sm_scale * kLog2e;
      mbar_wait(&bars[kLutFull + (n & 1)], (n >> 1) & 1);

      float m_used = -INFINITY, l_sum = 0.f;
      for (int j = 0; j < T_blocks; ++j, ++g) {
        const uint32_t sb = g & 1u;
        const int blk = s_lut[j];
        const float sc = qsc * s_ksc[j];
        const int valid = p.lk - blk * BLKK - hf * 32;   // columns of MY half that are real keys (>= 32: all)
        int mxa = -2147483647 - 1, mxb = mxa;
        const uint32_t ts = tmem_base + lane_addr + kColS + sb * BLKK + hf * 32;
        {
          uint32_t& par = sb ? s_par1 : s_par0;
          mbar_wait(&bars[kSFull + sb], par & 1u);
          ++par;
        }
        tc_fence_after_sync();
        // ---- pass 1 over my 32 scores: row maximum only (the registers are released; pass 2 reads tensor memory again in
        //      two 16-column pieces, which keeps the live set inside the 96 registers two co-resident CTAs allow)
        const uint32_t keep = valid >= 32 ? 0xFFFFFFFFu : (valid <= 0 ? 0u : ((1u << valid) - 1u));  // real key columns
        {
          uint32_t s[32];
          tmem_ld_x32(ts, s);
          tmem_ld_wait();
          if (valid < 32) {  // ragged last key block: masked columns count as INT_MIN
#pragma unroll
            for (int c = 0; c < 32; ++c)
              if (!((keep >> c) & 1u)) s[c] = 0x80000000u;
          }
#pragma unroll
          for (int c = 0; c < 32; c += 4) {
            mxa = __vimax3_s32(mxa, static_cast<int>(s[c]), static_cast<int>(s[c + 1]));
            mxb = __vimax3_s32(mxb, static_cast<int>(s[c + 2]), static_cast<int>(s[c + 3]));
          }
        }
        // ---- row maximum across the two halves of the row
        float* xm = x_max + (g & 1u) * 256;
        xm[hf * 128 + r] = static_cast<float>(max(mxa, mxb));
        named_bar_sync(pair_bar, 64);
        const float m_blk_f = fmaxf(xm[r], xm[128 + r]) * sc;

        // ---- lazy rescale of the O accumulator (both warps of the pair reach the same decision: same rows, same data)
        const bool grow = m_blk_f > m_used + kRescaleThreshold;
        if (j == 0) {
          m_used = m_blk_f;
        } else if (__any_sync(0xffffffffu, grow)) {
          const float m_new = grow ? m_blk_f : m_used;
          const float alpha = fast_exp2(m_used - m_new);
          while (pv_waited < p_pub) {                     // every P.V issued so far has retired
            mbar_wait(&bars[kPvDone], pv_waited & 1u);
            ++pv_waited;
          }
          tc_fence_after_sync();
          const uint32_t to = tmem_base + lane_addr + kColO + hf * (HD / 2);
#pragma unroll
          for (int c = 0; c < HD / 64; ++c) {
            uint32_t o[32];
            tmem_ld_x32(to + c * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_x32(to + c * 32, o);
          }
          tmem_st_wait();
          tc_fence_before_sync();
          l_sum *= alpha;
          m_used = m_new;
        }

        // ---- pass 2: P = exp2(s*sc - m_used) for my 32 columns, 16 at a time
        const float cbias = -fmaf(kMagicF, sc, m_used);
        const float2 sc2 = make_float2(sc, sc), cb2 = make_float2(cbias, cbias);
        float2 psa = make_float2(0.f, 0.f), psb = psa;
        uint32_t pw[16];
#pragma unroll
        for (int hc = 0; hc < 2; ++hc) {
          uint32_t s[16];
          tmem_ld_x16(ts + hc * 16, s);
          tmem_ld_wait();
          if (valid < 32) {
#pragma unroll
            for (int c = 0; c < 16; ++c)
              if (!((keep >> (hc * 16 + c)) & 1u)) s[c] = 0x80000000u;
          }
#pragma unroll
          for (int c = 0; c < 16; c += 4) {
            float2 t0 = __ffma2_rn(make_float2(__int_as_float(static_cast<int>(s[c]) + kMagicI),
                                               __int_as_float(static_cast<int>(s[c + 1]) + kMagicI)), sc2, cb2);
            float2 t1 = __ffma2_rn(make_float2(__int_as_float(static_cast<int>(s[c + 2]) + kMagicI),
                                               __int_as_float(static_cast<int>(s[c + 3]) + kMagicI)), sc2, cb2);
            t0.x = fast_exp2(t0.x); t0.y = fast_exp2(t0.y);
            t1.x = fast_exp2(t1.x); t1.y = fast_exp2(t1.y);
            psa = __fadd2_rn(psa, t0);
            psb = __fadd2_rn(psb, t1);
            pw[hc * 8 + (c >> 1)] = F16Traits<T>::pack(t0.x, t0.y);
            pw[hc * 8 + (c >> 1) + 1] = F16Traits<T>::pack(t1.x, t1.y);
          }
        }
        // P(j) of half hf goes to columns [16*hf, 16*hf+16) of this S buffer: half 1 stores over S columns [16, 32), which
        // half 0 reads in pass 2.  Both halves finish reading S before either stores P.
        tc_fence_before_sync();
        named_bar_sync(pair_bar, 64);
        const float2 ps2 = __fadd2_rn(psa, psb);
        float psum = ps2.x + ps2.y;
        if (valid < 32) {
          // exact fix-up of the ragged block: every masked column produced the same p (same INT_MIN input); remove it
          // from the row sum and clear its 16-bit slot so the tensor core multiplies V's zero-filled rows by zero
          const float pm = fast_exp2(fmaf(__int_as_float(static_cast<int>(0x80000000u) + kMagicI), sc, cbias));
          psum -= static_cast<float>(32 - __popc(keep)) * pm;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const uint32_t two = (keep >> (2 * i)) & 3u;   // bit 0: low half (even key) real, bit 1: high half real
            pw[i] &= (two & 1u ? 0x0000FFFFu : 0u) | (two & 2u ? 0xFFFF0000u : 0u);
          }
        }
        l_sum += psum;

        // ---- publish P(j): at most one P.V may be outstanding (keeps the PFull / PvDone phase parities unambiguous)
        while (pv_waited < p_pub) {
          mbar_wait(&bars[kPvDone], pv_waited & 1u);
          ++pv_waited;
        }
        tc_fence_after_sync();
        tmem_st_x16(tmem_base + lane_addr + kColS + sb * BLKK + hf * 16, pw);
        tmem_st_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[kPFull]);
        ++p_pub;
      }
      if (lane == 0) mbar_arrive(&bars[kLutFree + (n & 1)]);

      // ---- linear branch operand.  f_j = feature map numerator of my half of the query row (SLA/core.py:243):
      //      pass 1: E = sum f_j, F = sum f_j * ksum_j;  phi_j = f_j / E (softmax) or f_j;  den = 1e-5 + sum phi_j ksum_j
      //      pass 2: A_j = T(phi_j * l / den) -> tensor memory, so that O + A.KVW^T = l * (O/l + phi.KVW^T/den)
      const int64_t q_row = int64_t(m_blk) * BLKQ + r;
      const T* qrow = static_cast<const T*>(p.q) + ((int64_t(b) * p.l + (q_row < p.l ? q_row : p.l - 1)) * p.h + hh) * HD + hf * (HD / 2);
      constexpr int NW = HD / 4;                          // packed 32-bit words in my half row (HD/2 elements)
      uint32_t raw[NW];
#pragma unroll
      for (int c = 0; c < NW / 4; ++c) {
        const uint4 v4 = __ldg(reinterpret_cast<const uint4*>(qrow) + c);
        raw[4 * c] = v4.x; raw[4 * c + 1] = v4.y; raw[4 * c + 2] = v4.z; raw[4 * c + 3] = v4.w;
      }
      float* xs = x_sum;                                  // [0]: row max / l, [1]: E, [2]: F   each [2 half][128]
      float off = 0.f;
      if (p.feature == 0) {
        float qm = -INFINITY;
#pragma unroll
        for (int i = 0; i < NW; ++i) qm = fmaxf(qm, fmaxf(F16Traits<T>::lo(raw[i]), F16Traits<T>::hi(raw[i])));
        xs[hf * 128 + r] = qm;
        named_bar_sync(pair_bar, 64);
        off = fmaxf(xs[r], xs[128 + r]) * kLog2e;
        named_bar_sync(pair_bar, 64);                     // slot [0] is reused for l below
      }
      const float* ks = p.ksum + int64_t(bh) * HD + hf * (HD / 2);
      float e0 = 0.f, e1 = 0.f, f0 = 0.f, f1 = 0.f;
#pragma unroll
      for (int i = 0; i < NW; i += 2) {
        const float4 k4 = __ldg(reinterpret_cast<const float4*>(ks + 2 * i));
        const float a0 = feat<T>(F16Traits<T>::lo(raw[i]), off, p.feature), a1 = feat<T>(F16Traits<T>::hi(raw[i]), off, p.feature);
        const float a2 = feat<T>(F16Traits<T>::lo(raw[i + 1]), off, p.feature), a3 = feat<T>(F16Traits<T>::hi(raw[i + 1]), off, p.feature);
        e0 += a0 + a1;
        e1 += a2 + a3;
        f0 = fmaf(a0, k4.x, fmaf(a1, k4.y, f0));
        f1 = fmaf(a2, k4.z, fmaf(a3, k4.w, f1));
      }
      xs[hf * 128 + r] = l_sum;
      xs[256 + hf * 128 + r] = e0 + e1;
      xs[512 + hf * 128 + r] = f0 + f1;
      named_bar_sync(pair_bar, 64);
      const float l_tot = xs[r] + xs[128 + r];
      const float E = xs[256 + r] + xs[384 + r];
      const float F = xs[512 + r] + xs[640 + r];
      const float inv_e = p.feature == 0 ? 1.0f / E : 1.0f;
      const float den = 1e-5f + F * inv_e;
      const float cscale = inv_e * l_tot / den;
#pragma unroll
      for (int i = 0; i < NW; ++i)   // in place: raw q words become the packed A operand
        raw[i] = F16Traits<T>::pack(feat<T>(F16Traits<T>::lo(raw[i]), off, p.feature) * cscale,
                                    feat<T>(F16Traits<T>::hi(raw[i]), off, p.feature) * cscale);
      // slot g (= g0 + T): its S buffer last held P(T-2), whose P.V retired before P(T-1) was published
      {
        const uint32_t ta = tmem_base + lane_addr + kColS + (g & 1u) * BLKK + hf * NW;
        if constexpr (NW == 32) {
          tmem_st_x32(ta, raw);
        } else {
          tmem_st_x16(ta, raw);
        }
        tmem_st_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[kPhiFull]);
      }
      ++g;

      // ---- out = T( O / l + proj_b ) for my half of the row, straight from registers (one full 128-byte line per thread
      //      for HD = 128)
      mbar_wait(&bars[kOFull], n & 1);
      tc_fence_after_sync();
      const float inv_l = 1.0f / l_tot;
      T* orow = static_cast<T*>(p.out) + ((int64_t(b) * p.l + q_row) * p.h + hh) * HD + hf * (HD / 2);
      const float* pb = p.proj_b + hf * (HD / 2);
#pragma unroll
      for (int c = 0; c < HD / 64; ++c) {
        uint32_t o[32];
        tmem_ld_x32(tmem_base + lane_addr + kColO + hf * (HD / 2) + c * 32, o);
        tmem_ld_wait();
        if (c == HD / 64 - 1) {  // all of my O columns are in registers: the next tile's first P.V may overwrite O
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars[kOFree]);
        }
#pragma unroll
        for (int g4 = 0; g4 < 4; ++g4) {
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(pb + c * 32 + g4 * 8));
          const float4 b1 = __ldg(reinterpret_cast<const float4*>(pb + c * 32 + g4 * 8) + 1);
          uint4 w;
          w.x = F16Traits<T>::pack(fmaf(__uint_as_float(o[g4 * 8 + 0]), inv_l, b0.x), fmaf(__uint_as_float(o[g4 * 8 + 1]), inv_l, b0.y));
          w.y = F16Traits<T>::pack(fmaf(__uint_as_float(o[g4 * 8 + 2]), inv_l, b0.z), fmaf(__uint_as_float(o[g4 * 8 + 3]), inv_l, b0.w));
          w.z = F16Traits<T>::pack(fmaf(__uint_as_float(o[g4 * 8 + 4]), inv_l, b1.x), fmaf(__uint_as_float(o[g4 * 8 + 5]), inv_l, b1.y));
          w.w = F16Traits<T>::pack(fmaf(__uint_as_float(o[g4 * 8 + 6]), inv_l, b1.z), fmaf(__uint_as_float(o[g4 * 8 + 7]), inv_l, b1.w));
          if (q_row < p.l) stg_v4(orow + c * 32 + g4 * 8, w);
        }
      }
    }
    tc_fence_before_sync();
  }

  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

}  // namespace

template <int HD>
static int launch_v2(const int8_t* q_i8, const float* q_scale, const int8_t* k_i8, const float* k_scale, const void* v,
                     const void* q, int dtype, const int32_t* lut, int64_t topk, const void* kvw, const float* ksum,
                     const float* proj_b, void* out, int64_t b, int64_t l, int64_t lk, int64_t h, float sm_scale, int feature,
                     void* stream) {
  using namespace tdb;
  using C = Cfg<HD>;
  const int64_t d = HD;
  const int64_t mblk = cdiv64(l, BLKQ), nblk = cdiv64(lk, BLKK);
  const int64_t tiles = mblk * h * b;
  if (tiles > (int64_t(1) << 30)) return fail(TDB200_ERR_UNSUPPORTED, "sla_attn_fwd: too many tiles");
  const size_t lut_stride = (size_t(topk) * 6 + 15) & ~size_t(15);
  const size_t smem = 1024 + C::kOffLut + 2 * lut_stride;
  if (smem > 227 * 1024) return fail(TDB200_ERR_UNSUPPORTED, "sla_attn_fwd: topk=%lld too large for on-chip LUT", (long long)topk);

  const CUtensorMapDataType t16 = dtype == TDB200_DTYPE_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const int sw8 = HD == 128 ? 128 : 64;
  CUtensorMap tq, tk, tv, tw;
  {
    const uint64_t dims[4] = {uint64_t(d), uint64_t(l), uint64_t(b * h), 1};
    const uint64_t str[3] = {uint64_t(d), uint64_t(l * d), uint64_t(b * h * l * d)};
    const uint32_t box[4] = {uint32_t(HD), BLKQ, 1, 1};
    if (int rc = make_tmap_4d(&tq, q_i8, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, dims, str, box, sw8)) return rc;
  }
  {
    const uint64_t dims[4] = {uint64_t(d), uint64_t(lk), uint64_t(b * h), 1};
    const uint64_t str[3] = {uint64_t(d), uint64_t(lk * d), uint64_t(b * h * lk * d)};
    const uint32_t box[4] = {uint32_t(HD), BLKK, 1, 1};
    if (int rc = make_tmap_4d(&tk, k_i8, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, dims, str, box, sw8)) return rc;
  }
  {
    const uint64_t dims[4] = {uint64_t(d), uint64_t(h), uint64_t(lk), uint64_t(b)};
    const uint64_t str[3] = {uint64_t(d * 2), uint64_t(h * d * 2), uint64_t(lk * h * d * 2)};
    const uint32_t box[4] = {64, 1, BLKK, 1};
    if (int rc = make_tmap_4d(&tv, v, t16, 2, dims, str, box)) return rc;
  }
  {
    const uint64_t dims[4] = {uint64_t(d), uint64_t(d), uint64_t(b * h), 1};
    const uint64_t str[3] = {uint64_t(d * 2), uint64_t(d * d * 2), uint64_t(b * h * d * d * 2)};
    const uint32_t box[4] = {64, uint32_t(HD), 1, 1};
    if (int rc = make_tmap_4d(&tw, kvw, t16, 2, dims, str, box)) return rc;
  }
  AttnParams p;
  p.q_scale = q_scale;
  p.k_scale = k_scale;
  p.q = q;
  p.lut = lut;
  p.ksum = ksum;
  p.proj_b = proj_b;
  p.out = out;
  p.l = int(l);
  p.lk = int(lk);
  p.h = int(h);
  p.mblk = int(mblk);
  p.nblk = int(nblk);
  p.topk = int(topk);
  p.tiles = int(tiles);
  p.feature = feature;
  p.sm_scale = sm_scale;
  int grid = 2 * sm_count();
  if (grid > tiles) grid = int(tiles);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define TDB_ATTN(T)                                                                                                   \
  do {                                                                                                                \
    if (int rc = check_cuda(cudaFuncSetAttribute(sla_attn_v2_kernel<T, HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                 static_cast<int>(smem)), "cudaFuncSetAttribute(sla_attn_v2)"))      \
      return rc;                                                                                                      \
    sla_attn_v2_kernel<T, HD><<<grid, kThreads, smem, st>>>(tq, tk, tv, tw, p);                                      \
    return check_launch("sla_attn_v2_kernel");                                                                        \
  } while (0)
  if (dtype == TDB200_DTYPE_BF16) TDB_ATTN(__nv_bfloat16);
  if (dtype == TDB200_DTYPE_FP16) TDB_ATTN(__half);
#undef TDB_ATTN
  return fail(TDB200_ERR_UNSUPPORTED, "sla_attn_fwd: dtype tag %d", dtype);
}

extern "C" int tdb200_sla_attn_fwd_v2(const int8_t* q_i8, const float* q_scale, const int8_t* k_i8, const float* k_scale,
                                      const void* v, const void* q, int dtype, const int32_t* lut, int64_t topk,
                                      const void* kvw, const float* ksum, const float* proj_b, void* out, int64_t b,
                                      int64_t l, int64_t lk, int64_t h, int64_t d, float sm_scale, int feature,
                                      void* stream) {
  using namespace tdb;
  if (!q_i8 || !q_scale || !k_i8 || !k_scale || !v || !q || !lut || !kvw || !ksum || !proj_b || !out)
    return fail(TDB200_ERR_INVALID_ARG, "sla_attn_fwd: null pointer");
  if (b <= 0 || l <= 0 || lk <= 0 || h <= 0) return fail(TDB200_ERR_INVALID_ARG, "sla_attn_fwd: bad shape");
  if (d != 64 && d != 128) return fail(TDB200_ERR_UNSUPPORTED, "sla_attn_fwd: head dim %lld (64 or 128, SLA/core.py:207)", (long long)d);
  if (feature < 0 || feature > 2) return fail(TDB200_ERR_INVALID_ARG, "sla_attn_fwd: feature map tag %d", feature);
  const int64_t nblk = cdiv64(lk, BLKK);
  if (topk <= 0 || topk > nblk) return fail(TDB200_ERR_INVALID_ARG, "sla_attn_fwd: topk=%lld outside [1, %lld]", (long long)topk, (long long)nblk);
  if (nblk > 65535 || h > 65535 || b > 65535) return fail(TDB200_ERR_UNSUPPORTED, "sla_attn_fwd: dimension too large");
  if (int rc = require_sm100()) return rc;
  if (d == 128)
    return launch_v2<128>(q_i8, q_scale, k_i8, k_scale, v, q, dtype, lut, topk, kvw, ksum, proj_b, out, b, l, lk, h, sm_scale, feature, stream);
  return launch_v2<64>(q_i8, q_scale, k_i8, k_scale, v, q, dtype, lut, topk, kvw, ksum, proj_b, out, b, l, lk, h, sm_scale, feature, stream);
}
