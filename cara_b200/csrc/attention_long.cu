// Attention core of cp_attn (cara.py:44-48) on the 5th-generation tensor cores for D = 64 and N > 256 tokens
// (ViT-B/L/16 fine-tuned at 384 px: N = 577; 448 px: N = 785).  The N <= 256 kernels of attention_tc.cu hold a whole
// head in shared memory; these kernels tile the keys (forward, dQ) or the queries (dK / dV) in 128-row blocks and
// stream them through a two-stage TMA ring, so shared memory does not grow with N.
//
// Q, K, V are read with one TMA map straight out of the fused projection's [B*N, 3*H*64] output (128-row boxes, 128-byte
// swizzle), dO with a second map over [B*N, H*64].  A box that starts inside sample b runs into sample b+1 (or past the
// end of the tensor, where TMA fills zeros); every such row is masked by index: keys >= N get p = 0 (-inf before the
// max), query rows >= N get P = dS = 0 in the backward, and no row >= N is ever stored.
//
//   attn_fwd_long_kernel   work item (sample, head, 128-query tile); persistent CTAs, TWO per SM.  Per key tile j:
//                          S_j = Q K_j^T -> TMEM (128 columns), online max / sum in the softmax thread that owns the
//                          query row, P_j packed bf16 over the consumed scores, O_j = P_j V_j (A = P from TMEM, B = V
//                          MN-major) into the consumed upper half of the same 128 columns; the thread folds
//                          O <- alpha O + O_j in 64 fp32 registers.  S is double-buffered so Q K_{j+1}^T overlaps the
//                          softmax of tile j.  TMEM: 2 x 128 columns (S_j / P_j / O_j) = 256 per CTA, 512 per SM.
//   attn_bwd_dkdv_kernel   work item (sample, head, 128-key tile); one CTA per SM.  K_j, V_j resident; Q_i, dO_i stream.
//                          S^T = K_j Q_i^T, dP^T = V_j dO_i^T (keys on the TMEM lanes), P^T = 2^(S^T sl2 - lse),
//                          dS^T = P^T (.) (dP^T - delta); dV += P^T dO_i (P^T from TMEM), dK += dS^T Q_i (dS^T through
//                          one 32 KB swizzled shared tile).  TMEM: 128 + 128 + 64 + 64 = 384 of 512 columns.
//   attn_bwd_dq_kernel     work item (sample, head, 128-query tile); one CTA per SM.  Q_i, dO_i resident; K_j, V_j
//                          stream.  S, dP recomputed, dS packed bf16 into TMEM over the consumed scores,
//                          dQ += dS K_j (A = dS from TMEM, B = K_j MN-major).  TMEM: 128 + 128 + 64 = 320 of 512.
// Every dqkv element is written by exactly one thread of one CTA and summed in a fixed order: no atomics, so the
// backward is bit-identical from run to run.
#include "gemm_sm100.h"
#include "kernels.h"
#include "ptx.cuh"

#include <math_constants.h>

namespace cara {
namespace {

constexpr int LD = 64;                    // head dim
constexpr uint32_t TB = 16384;            // one 128-row x 64-column bf16 tile
constexpr float LOG2E = 1.4426950408889634f;

// ------------------------------------------------------------------------------------ forward
constexpr int LF_THREADS = 192;           // warps 0-3: softmax / epilogue (thread = query row = TMEM lane), 4: MMA, 5: TMA
constexpr int LF_TMEM_COLS = 256;

__global__ void __launch_bounds__(LF_THREADS, 2)
attn_fwd_long_kernel(const __grid_constant__ CUtensorMap map_qkv, const AttnArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t sQ = (raw + 1023u) & ~1023u;
  const uint32_t ring = sQ + TB;                                // stage s: K at ring + 2s TB, V at ring + (2s+1) TB
  const uint32_t bars = ring + 4u * TB;
  const uint32_t bar_full = bars, bar_empty = bars + 16, bar_s = bars + 32, bar_p = bars + 48, bar_o = bars + 64,
                 bar_free = bars + 80, bar_qfull = bars + 96, bar_qempty = bars + 104, tmem_slot = bars + 112;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N, C = a.H * LD;
  const int nt = (N + 127) / 128;
  const int items = a.B * a.H * nt;

  if (warp == 4) {
    if (lane == 0) {
      tma_prefetch_desc(&map_qkv);
      for (int s = 0; s < 2; ++s) {
        mbar_init(bar_full + 8 * s, 1);
        mbar_init(bar_empty + 8 * s, 1);
        mbar_init(bar_s + 8 * s, 1);
        mbar_init(bar_p + 8 * s, 128);
        mbar_init(bar_o + 8 * s, 1);
        mbar_init(bar_free + 8 * s, 128);
      }
      mbar_init(bar_qfull, 1);
      mbar_init(bar_qempty, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc<LF_TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();                                                  // nothing above touches global memory
  pdl_trigger();

  if (warp == 5) {
    if (lane == 0) {
      uint32_t g = 0, it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const int bh = item / nt, qt = item % nt;
        const int row0 = (bh / a.H) * N, col = (bh % a.H) * LD;
        mbar_wait(bar_qempty, (it & 1u) ^ 1u);
        mbar_expect_tx(bar_qfull, TB);
        tma_load_2d(sQ, &map_qkv, bar_qfull, col, row0 + qt * 128);
        for (int j = 0; j < nt; ++j, ++g) {
          const uint32_t s = g & 1u;
          mbar_wait(bar_empty + 8u * s, ((g >> 1) & 1u) ^ 1u);
          mbar_expect_tx(bar_full + 8u * s, 2u * TB);
          tma_load_2d(ring + 2u * s * TB, &map_qkv, bar_full + 8u * s, C + col, row0 + j * 128);
          tma_load_2d(ring + (2u * s + 1u) * TB, &map_qkv, bar_full + 8u * s, 2 * C + col, row0 + j * 128);
        }
      }
    }
  } else if (warp == 4) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16_major(128, 128, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16_major(128, LD, 0, 1);
      // O_t = P_t V: P in the low 64 columns of buffer t & 1, O_t into its (consumed) high 64 columns
      auto pv = [&](uint32_t t, uint32_t g) {
        const uint32_t buf = t & 1u, sV = ring + (2u * (g & 1u) + 1u) * TB;
        mbar_wait(bar_p + 8u * buf, (t >> 1) & 1u);
        tc_fence_after();
        const uint32_t d = tmem_base + 128u * buf;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          umma_bf16_ts(d + 64u, d + 8u * k, umma_desc_mn_sw128(sV + static_cast<uint32_t>(k) * 2048u, TB, 1024u), idesc_o,
                       k != 0 ? 1u : 0u);
        umma_commit(bar_o + 8u * buf);
        umma_commit(bar_empty + 8u * (g & 1u));                // K_j / V_j are dead
      };
      uint32_t g = 0, t = 0, it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        mbar_wait(bar_qfull, it & 1u);
        for (int j = 0; j < nt; ++j, ++g, ++t) {
          const uint32_t s = g & 1u, buf = t & 1u;
          mbar_wait(bar_full + 8u * s, (g >> 1) & 1u);
          mbar_wait(bar_free + 8u * buf, ((t >> 1) & 1u) ^ 1u);  // O_{t-2} has been read out of this buffer
          tc_fence_after();
          const uint64_t dq = umma_desc_sw128(sQ), dk = umma_desc_sw128(ring + 2u * s * TB);
#pragma unroll
          for (int k = 0; k < LD / 16; ++k)
            umma_bf16(tmem_base + 128u * buf, dq + 2u * k, dk + 2u * k, idesc_s, k != 0 ? 1u : 0u);
          umma_commit(bar_s + 8u * buf);
          if (j == nt - 1) umma_commit(bar_qempty);             // Q is dead once the item's last S has retired
          if (j > 0) pv(t - 1, g - 1);                          // S_{j} overlaps the softmax of tile j - 1
        }
        pv(t - 1, g - 1);
      }
    }
  } else {
    const int tq = warp * 32 + lane;                           // query row inside the tile = TMEM lane
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    const float sl2 = a.scale * LOG2E;
    uint32_t t = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int bh = item / nt, qt = item % nt;
      const int b = bh / a.H, h = bh % a.H;
      const int row = qt * 128 + tq;
      float o[64];
#pragma unroll
      for (int e = 0; e < 64; ++e) o[e] = 0.f;
      float m = -CUDART_INF_F, l = 0.f;                        // running max (scaled, base 2) and sum
      for (int j = 0; j < nt; ++j, ++t) {
        const uint32_t buf = t & 1u, ph = (t >> 1) & 1u;
        const uint32_t sa = lane_addr + 128u * buf;
        const int nv = N - j * 128;                            // valid keys in this tile (>= 1)
        mbar_wait(bar_s + 8u * buf, ph);
        tc_fence_after();
        // pass 1: maximum over the valid keys
        float mx = -CUDART_INF_F;
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(sa + c0, r);
          tmem_ld_wait();
          if (c0 + 32 <= nv) {
#pragma unroll
            for (int e = 0; e < 32; ++e) mx = fmaxf(mx, __uint_as_float(r[e]));
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e) if (c0 + e < nv) mx = fmaxf(mx, __uint_as_float(r[e]));
          }
        }
        const float mn = fmaxf(m, mx * sl2);                   // finite: every tile holds a valid key
        const float alpha = exp2f(m - mn);                     // 0 on the first tile
        // pass 2: p = 2^(s sl2 - mn), tile sum, packed bf16 over the consumed scores (columns c0/2 .. c0/2 + 15)
        float lt = 0.f;
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          uint32_t r[32], pk[16];
          tmem_ld32(sa + c0, r);
          tmem_ld_wait();
          if (c0 + 32 <= nv) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const float p0 = exp2f(fmaf(__uint_as_float(r[2 * e]), sl2, -mn));
              const float p1 = exp2f(fmaf(__uint_as_float(r[2 * e + 1]), sl2, -mn));
              lt += p0 + p1;
              pk[e] = pack_bf16(p0, p1);
            }
          } else {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              float p0 = exp2f(fmaf(__uint_as_float(r[2 * e]), sl2, -mn));
              float p1 = exp2f(fmaf(__uint_as_float(r[2 * e + 1]), sl2, -mn));
              if (c0 + 2 * e >= nv) p0 = 0.f;
              if (c0 + 2 * e + 1 >= nv) p1 = 0.f;
              lt += p0 + p1;
              pk[e] = pack_bf16(p0, p1);
            }
          }
          tmem_st16(sa + (c0 >> 1), pk);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(bar_p + 8u * buf);
        mbar_wait(bar_o + 8u * buf, ph);
        tc_fence_after();
        uint32_t r0[32], r1[32];
        tmem_ld32(sa + 64u, r0);
        tmem_ld32(sa + 96u, r1);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(bar_free + 8u * buf);
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          o[e] = fmaf(o[e], alpha, __uint_as_float(r0[e]));
          o[32 + e] = fmaf(o[32 + e], alpha, __uint_as_float(r1[e]));
        }
        l = fmaf(l, alpha, lt);
        m = mn;
      }
      if (row < N) {
        const float inv = 1.0f / l;
        const long off = (static_cast<long>(b) * N + row) * C + h * LD;
        __nv_bfloat16* po = a.o + off;
        __nv_bfloat16* pl = a.o_lo != nullptr ? a.o_lo + off : nullptr;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float v0 = o[16 * j + 2 * e] * inv, v1 = o[16 * j + 2 * e + 1] * inv;
            hi[e] = pack_bf16(v0, v1);
            const float2 hf = unpack_bf16(hi[e]);
            lo[e] = pack_bf16(v0 - hf.x, v1 - hf.y);
          }
          st_global_v8(po + 16 * j, hi);
          if (pl != nullptr) st_global_v8(pl + 16 * j, lo);
        }
        if (a.lse != nullptr) a.lse[(static_cast<long>(b) * a.H + h) * N + row] = m + log2f(l);
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc<LF_TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------ backward
// Both backward kernels: warps 0-7 compute (TMEM lane quarter = warp & 3, column half = warp >> 2: each half takes 64 of
// the 128 score columns and packs its bf16 results into the first 32 columns of its own, consumed range, so k-step
// kk of the packed operand sits at column 8 kk + 32 [kk >= 4]), warp 8 issues the MMAs, warp 9 the TMA loads.
constexpr int LB_THREADS = 320;
constexpr int LB_DP_COL = 128, LB_ACC_COL = 256;

__device__ __forceinline__ uint32_t packed_col(int kk) { return static_cast<uint32_t>(8 * kk + (kk >= 4 ? 32 : 0)); }
__device__ __forceinline__ void compute_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// barrier block shared by the two backward kernels
struct BwdBars {
  uint32_t full, empty, res_full, res_empty, sdp, p, mma, acc_free, tmem_slot;
  __device__ explicit BwdBars(uint32_t base)
      : full(base), empty(base + 16), res_full(base + 32), res_empty(base + 40), sdp(base + 48), p(base + 56),
        mma(base + 64), acc_free(base + 72), tmem_slot(base + 80) {}
  __device__ void init(int compute_threads) const {
    for (int s = 0; s < 2; ++s) {
      mbar_init(full + 8 * s, 1);
      mbar_init(empty + 8 * s, 1);
    }
    mbar_init(res_full, 1);
    mbar_init(res_empty, 1);
    mbar_init(sdp, 1);
    mbar_init(p, compute_threads);
    mbar_init(mma, 1);
    mbar_init(acc_free, compute_threads);
    fence_mbar_init();
  }
};

// dK / dV.  TMEM: S^T [0,128), dP^T [128,256), dV [256,320), dK [320,384).
__global__ void __launch_bounds__(LB_THREADS, 1)
attn_bwd_dkdv_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do,
                     const AttnArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t sK = (raw + 1023u) & ~1023u, sV = sK + TB;
  const uint32_t ring = sV + TB;                                // stage s: Q at ring + 2s TB, dO at ring + (2s+1) TB
  const uint32_t sDS = ring + 4u * TB;                          // dS^T: [64-query block][128 keys][128 B], swizzled
  const uint32_t stats = sDS + 2u * TB;                         // [2 buffers][-lse 128 | delta 128] fp32
  const BwdBars bb(stats + 2048u);
  float* s_stats = reinterpret_cast<float*>(smem_raw + (stats - raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (bb.tmem_slot - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N, C = a.H * LD;
  const int nt = (N + 127) / 128;
  const int items = a.B * a.H * nt;

  if (warp == 8) {
    if (lane == 0) {
      tma_prefetch_desc(&map_qkv);
      tma_prefetch_desc(&map_do);
      bb.init(256);
    }
    __syncwarp();
    tmem_alloc<512>(bb.tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();
  pdl_trigger();

  if (warp == 9) {
    if (lane == 0) {
      uint32_t g = 0, it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const int bh = item / nt, kt = item % nt;
        const int row0 = (bh / a.H) * N, col = (bh % a.H) * LD;
        mbar_wait(bb.res_empty, (it & 1u) ^ 1u);
        mbar_expect_tx(bb.res_full, 2u * TB);
        tma_load_2d(sK, &map_qkv, bb.res_full, C + col, row0 + kt * 128);
        tma_load_2d(sV, &map_qkv, bb.res_full, 2 * C + col, row0 + kt * 128);
        for (int i = 0; i < nt; ++i, ++g) {
          const uint32_t s = g & 1u;
          mbar_wait(bb.empty + 8u * s, ((g >> 1) & 1u) ^ 1u);
          mbar_expect_tx(bb.full + 8u * s, 2u * TB);
          tma_load_2d(ring + 2u * s * TB, &map_qkv, bb.full + 8u * s, col, row0 + i * 128);
          tma_load_2d(ring + (2u * s + 1u) * TB, &map_do, bb.full + 8u * s, col, row0 + i * 128);
        }
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16_major(128, 128, 0, 0);
      constexpr uint32_t idesc_acc = umma_idesc_bf16_major(128, LD, 0, 1);   // A K-major (TMEM / smem), B MN-major
      uint32_t g = 0, n = 0, it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        mbar_wait(bb.res_full, it & 1u);
        for (int i = 0; i < nt; ++i, ++g, ++n) {
          const uint32_t s = g & 1u;
          const uint32_t sQ = ring + 2u * s * TB, sDO = sQ + TB;
          mbar_wait(bb.full + 8u * s, (g >> 1) & 1u);
          if (n > 0) mbar_wait(bb.mma, (n - 1u) & 1u);          // P^T / dS^T of the previous tile have been consumed
          tc_fence_after();
          {
            const uint64_t dk = umma_desc_sw128(sK), dq = umma_desc_sw128(sQ);
            const uint64_t dv = umma_desc_sw128(sV), dd = umma_desc_sw128(sDO);
#pragma unroll
            for (int k = 0; k < LD / 16; ++k) umma_bf16(tmem_base, dk + 2u * k, dq + 2u * k, idesc_s, k != 0 ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < LD / 16; ++k)
              umma_bf16(tmem_base + LB_DP_COL, dv + 2u * k, dd + 2u * k, idesc_s, k != 0 ? 1u : 0u);
          }
          umma_commit(bb.sdp);
          if (i == 0 && it > 0) mbar_wait(bb.acc_free, (it - 1u) & 1u);   // the previous item's dK / dV were read out
          mbar_wait(bb.p, n & 1u);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const uint32_t acc = (i > 0 || kk > 0) ? 1u : 0u;
            umma_bf16_ts(tmem_base + LB_ACC_COL, tmem_base + packed_col(kk),
                         umma_desc_mn_sw128(sDO + static_cast<uint32_t>(kk) * 2048u, TB, 1024u), idesc_acc, acc);
            umma_bf16(tmem_base + LB_ACC_COL + 64u,
                      umma_desc_sw128(sDS + static_cast<uint32_t>(kk >> 2) * TB + static_cast<uint32_t>(kk & 3) * 32u),
                      umma_desc_mn_sw128(sQ + static_cast<uint32_t>(kk) * 2048u, TB, 1024u), idesc_acc, acc);
          }
          umma_commit(bb.mma);
          umma_commit(bb.empty + 8u * s);                       // Q_i / dO_i are dead
          if (i == nt - 1) umma_commit(bb.res_empty);           // so are K_j / V_j after the item's last tile
        }
      }
    }
  } else {
    const int q4 = warp & 3, half = warp >> 2, tid = threadIdx.x;
    const int key_local = q4 * 32 + lane;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const float sl2 = a.scale * LOG2E;
    const uint32_t ds_row = sDS + static_cast<uint32_t>(key_local) * 128u;
    const uint32_t sw = static_cast<uint32_t>(key_local & 7);
    const int cb = half * 64;
    uint32_t n = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int bh = item / nt, kt = item % nt;
      const int b = bh / a.H, h = bh % a.H;
      const long sbase = static_cast<long>(bh) * N;
      for (int i = 0; i < nt; ++i, ++n) {
        // statistics of query tile i (columns); rows >= N get -lse = -1e30, delta = 0: P = dS = 0
        float* st = s_stats + 256 * (n & 1u);
        {
          const int q = i * 128 + (tid & 127);
          if (tid < 128) st[tid] = q < N ? -a.lse[sbase + q] : -1e30f;
          else st[tid] = q < N ? a.delta[sbase + q] : 0.f;
        }
        compute_bar_sync();
        mbar_wait(bb.sdp, n & 1u);
        tc_fence_after();
#pragma unroll 1
        for (int c = cb; c < cb + 64; c += 16) {
          uint32_t s[16], dp[16], pk[8], dsk[8];
          tmem_ld16(lane_addr + c, s);
          tmem_ld16(lane_addr + LB_DP_COL + c, dp);
          tmem_ld_wait();
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 L = *reinterpret_cast<const float4*>(st + c + 4 * j4);
            const float4 Dl = *reinterpret_cast<const float4*>(st + 128 + c + 4 * j4);
            const float p0 = exp2f(fmaf(__uint_as_float(s[4 * j4 + 0]), sl2, L.x));
            const float p1 = exp2f(fmaf(__uint_as_float(s[4 * j4 + 1]), sl2, L.y));
            const float p2 = exp2f(fmaf(__uint_as_float(s[4 * j4 + 2]), sl2, L.z));
            const float p3 = exp2f(fmaf(__uint_as_float(s[4 * j4 + 3]), sl2, L.w));
            const float d0 = p0 * (__uint_as_float(dp[4 * j4 + 0]) - Dl.x);
            const float d1 = p1 * (__uint_as_float(dp[4 * j4 + 1]) - Dl.y);
            const float d2 = p2 * (__uint_as_float(dp[4 * j4 + 2]) - Dl.z);
            const float d3 = p3 * (__uint_as_float(dp[4 * j4 + 3]) - Dl.w);
            pk[2 * j4] = pack_bf16(p0, p1); pk[2 * j4 + 1] = pack_bf16(p2, p3);
            dsk[2 * j4] = pack_bf16(d0, d1); dsk[2 * j4 + 1] = pack_bf16(d2, d3);
          }
          tmem_st8(lane_addr + static_cast<uint32_t>(cb + ((c - cb) >> 1)), pk);
          const uint32_t blk = ds_row + static_cast<uint32_t>(c >> 6) * TB;
          const uint32_t ch = static_cast<uint32_t>((c & 63) >> 3);
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(blk + ((ch ^ sw) << 4)), "r"(dsk[0]), "r"(dsk[1]),
                       "r"(dsk[2]), "r"(dsk[3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(blk + (((ch + 1u) ^ sw) << 4)), "r"(dsk[4]),
                       "r"(dsk[5]), "r"(dsk[6]), "r"(dsk[7]) : "memory");
        }
        tmem_st_wait();
        fence_proxy_async();                                    // dS^T stores -> visible to the tensor core
        tc_fence_before();
        mbar_arrive(bb.p);
      }
      // read out: half 0 -> dK rows (scaled), half 1 -> dV rows; keys >= N are not stored
      mbar_wait(bb.mma, (n - 1u) & 1u);
      tc_fence_after();
      const int key = kt * 128 + key_local;
      const uint32_t col = LB_ACC_COL + (half == 0 ? 64u : 0u);
      const float sc = half == 0 ? a.scale : 1.0f;
      __nv_bfloat16* dst = a.dqkv + (static_cast<long>(b) * N + key) * 3 * C + (half == 0 ? C : 2 * C) + h * LD;
#pragma unroll
      for (int part = 0; part < 2; ++part) {
        uint32_t r[32];
        tmem_ld32(lane_addr + col + 32 * part, r);
        tmem_ld_wait();
        if (key < N) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            uint32_t w[8];
#pragma unroll
            for (int e = 0; e < 8; ++e)
              w[e] = pack_bf16(__uint_as_float(r[16 * j + 2 * e]) * sc, __uint_as_float(r[16 * j + 2 * e + 1]) * sc);
            st_global_v8(dst + 32 * part + 16 * j, w);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bb.acc_free);
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// dQ.  TMEM: S [0,128), dP [128,256), dQ [256,320).
__global__ void __launch_bounds__(LB_THREADS, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do,
                   const AttnArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t sQ = (raw + 1023u) & ~1023u, sDO = sQ + TB;
  const uint32_t ring = sDO + TB;                               // stage s: K at ring + 2s TB, V at ring + (2s+1) TB
  const BwdBars bb(ring + 4u * TB);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (bb.tmem_slot - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N, C = a.H * LD;
  const int nt = (N + 127) / 128;
  const int items = a.B * a.H * nt;

  if (warp == 8) {
    if (lane == 0) {
      tma_prefetch_desc(&map_qkv);
      tma_prefetch_desc(&map_do);
      bb.init(256);
    }
    __syncwarp();
    tmem_alloc<512>(bb.tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();
  pdl_trigger();

  if (warp == 9) {
    if (lane == 0) {
      uint32_t g = 0, it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const int bh = item / nt, qt = item % nt;
        const int row0 = (bh / a.H) * N, col = (bh % a.H) * LD;
        mbar_wait(bb.res_empty, (it & 1u) ^ 1u);
        mbar_expect_tx(bb.res_full, 2u * TB);
        tma_load_2d(sQ, &map_qkv, bb.res_full, col, row0 + qt * 128);
        tma_load_2d(sDO, &map_do, bb.res_full, col, row0 + qt * 128);
        for (int j = 0; j < nt; ++j, ++g) {
          const uint32_t s = g & 1u;
          mbar_wait(bb.empty + 8u * s, ((g >> 1) & 1u) ^ 1u);
          mbar_expect_tx(bb.full + 8u * s, 2u * TB);
          tma_load_2d(ring + 2u * s * TB, &map_qkv, bb.full + 8u * s, C + col, row0 + j * 128);
          tma_load_2d(ring + (2u * s + 1u) * TB, &map_qkv, bb.full + 8u * s, 2 * C + col, row0 + j * 128);
        }
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16_major(128, 128, 0, 0);
      constexpr uint32_t idesc_dq = umma_idesc_bf16_major(128, LD, 0, 1);   // A = dS from TMEM, B = K MN-major
      uint32_t g = 0, n = 0, it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        mbar_wait(bb.res_full, it & 1u);
        for (int j = 0; j < nt; ++j, ++g, ++n) {
          const uint32_t s = g & 1u;
          const uint32_t sK = ring + 2u * s * TB, sV = sK + TB;
          mbar_wait(bb.full + 8u * s, (g >> 1) & 1u);
          if (n > 0) mbar_wait(bb.mma, (n - 1u) & 1u);          // dS of the previous tile has been consumed
          tc_fence_after();
          {
            const uint64_t dq = umma_desc_sw128(sQ), dk = umma_desc_sw128(sK);
            const uint64_t dd = umma_desc_sw128(sDO), dv = umma_desc_sw128(sV);
#pragma unroll
            for (int k = 0; k < LD / 16; ++k) umma_bf16(tmem_base, dq + 2u * k, dk + 2u * k, idesc_s, k != 0 ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < LD / 16; ++k)
              umma_bf16(tmem_base + LB_DP_COL, dd + 2u * k, dv + 2u * k, idesc_s, k != 0 ? 1u : 0u);
          }
          umma_commit(bb.sdp);
          if (j == nt - 1) umma_commit(bb.res_empty);           // Q_i / dO_i are dead once the last S / dP retire
          if (j == 0 && it > 0) mbar_wait(bb.acc_free, (it - 1u) & 1u);   // the previous item's dQ was read out
          mbar_wait(bb.p, n & 1u);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_bf16_ts(tmem_base + LB_ACC_COL, tmem_base + packed_col(kk),
                         umma_desc_mn_sw128(sK + static_cast<uint32_t>(kk) * 2048u, TB, 1024u), idesc_dq,
                         (j > 0 || kk > 0) ? 1u : 0u);
          umma_commit(bb.mma);
          umma_commit(bb.empty + 8u * s);                       // K_j / V_j are dead
        }
      }
    }
  } else {
    const int q4 = warp & 3, half = warp >> 2;
    const int q_local = q4 * 32 + lane;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const float sl2 = a.scale * LOG2E;
    const int cb = half * 64;
    uint32_t n = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int bh = item / nt, qt = item % nt;
      const int b = bh / a.H, h = bh % a.H;
      const int q = qt * 128 + q_local;
      // query rows >= N: P = dS = 0
      const float nlse = q < N ? -a.lse[static_cast<long>(bh) * N + q] : -1e30f;
      const float dl = q < N ? a.delta[static_cast<long>(bh) * N + q] : 0.f;
      for (int j = 0; j < nt; ++j, ++n) {
        const int nv = N - j * 128;                            // valid keys in this tile
        mbar_wait(bb.sdp, n & 1u);
        tc_fence_after();
#pragma unroll 1
        for (int c = cb; c < cb + 64; c += 16) {
          uint32_t s[16], dp[16], dsk[8];
          tmem_ld16(lane_addr + c, s);
          tmem_ld16(lane_addr + LB_DP_COL + c, dp);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float p0 = exp2f(fmaf(__uint_as_float(s[2 * e]), sl2, nlse));
            float p1 = exp2f(fmaf(__uint_as_float(s[2 * e + 1]), sl2, nlse));
            if (c + 2 * e >= nv) p0 = 0.f;
            if (c + 2 * e + 1 >= nv) p1 = 0.f;
            dsk[e] = pack_bf16(p0 * (__uint_as_float(dp[2 * e]) - dl), p1 * (__uint_as_float(dp[2 * e + 1]) - dl));
          }
          tmem_st8(lane_addr + static_cast<uint32_t>(cb + ((c - cb) >> 1)), dsk);
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(bb.p);
      }
      // read out: each half stores 32 of the 64 columns of its query row
      mbar_wait(bb.mma, (n - 1u) & 1u);
      tc_fence_after();
      uint32_t r[32];
      tmem_ld32(lane_addr + LB_ACC_COL + 32u * half, r);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(bb.acc_free);
      if (q < N) {
        __nv_bfloat16* dst = a.dqkv + (static_cast<long>(b) * N + q) * 3 * C + h * LD + 32 * half;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          uint32_t w[8];
#pragma unroll
          for (int e = 0; e < 8; ++e)
            w[e] = pack_bf16(__uint_as_float(r[16 * j + 2 * e]) * a.scale, __uint_as_float(r[16 * j + 2 * e + 1]) * a.scale);
          st_global_v8(dst + 16 * j, w);
        }
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

int num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        sms <= 0)
      sms = 148;
  }
  return sms;
}

constexpr int LF_SMEM = 1024 + 5 * static_cast<int>(TB) + 128;
constexpr int LDKDV_SMEM = 1024 + 8 * static_cast<int>(TB) + 2048 + 128;
// 96 KB would be enough; asking for more than half of the SM's shared memory keeps this kernel at one CTA per SM, so
// its 512-column TMEM allocation never waits for a second resident CTA
constexpr int LDQ_SMEM = 120 * 1024;

}  // namespace

// D = 64, N > 256.  0 = launched, 1 = shape not covered, < 0 = error.
int attn_fwd_long_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.D != LD || a.N <= 256) return 1;
  const long rows = static_cast<long>(a.B) * a.N, cols = 3L * a.H * LD;
  CUtensorMap map;
  if (make_map_bf16(&map, a.qkv, rows, cols, cols, 128) != 0) return -54;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(attn_fwd_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LF_SMEM) != cudaSuccess)
      return -52;
    configured = true;
  }
  const long items = rows / a.N * a.H * ((a.N + 127) / 128);
  const int grid = static_cast<int>(items < 2L * num_sms() ? items : 2L * num_sms());
  return launch_pdl_f<2>(attn_fwd_long_kernel, dim3(grid), dim3(LF_THREADS), LF_SMEM, st, map, a) == cudaSuccess ? 0 : -53;
}

int attn_bwd_long_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.D != LD || a.N <= 256 || a.delta == nullptr) return 1;
  const long rows = static_cast<long>(a.B) * a.N, C = static_cast<long>(a.H) * LD;
  CUtensorMap map_qkv, map_do;
  if (make_map_bf16(&map_qkv, a.qkv, rows, 3 * C, 3 * C, 128) != 0) return -54;
  if (make_map_bf16(&map_do, a.d_o, rows, C, C, 128) != 0) return -54;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(attn_bwd_dkdv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LDKDV_SMEM) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LDQ_SMEM) != cudaSuccess)
      return -52;
    configured = true;
  }
  // a.o == nullptr: delta was written by the output projection's dX GEMM (EPI_DELTA), no pre-pass
  if (a.o != nullptr) {
    const int rc = attn_delta_launch(a, st);
    if (rc != 0) return rc;
  }
  const long items = static_cast<long>(a.B) * a.H * ((a.N + 127) / 128);
  const int grid = static_cast<int>(items < num_sms() ? items : num_sms());
  if (launch_pdl_f<2>(attn_bwd_dkdv_kernel, dim3(grid), dim3(LB_THREADS), LDKDV_SMEM, st, map_qkv, map_do, a) != cudaSuccess)
    return -53;
  return launch_pdl_f<2>(attn_bwd_dq_kernel, dim3(grid), dim3(LB_THREADS), LDQ_SMEM, st, map_qkv, map_do, a) == cudaSuccess
             ? 0 : -53;
}

}  // namespace cara
