// Attention core of cp_attn (cara.py:44-48) on the 5th-generation tensor cores: softmax(q k^T D^-1/2) v for
// D = 64 and N <= 256 tokens (ViT-B/L @224/16: N = 197), one CTA per (sample, head), two CTAs per SM.
//
//   TMA      : the head's Q, K, V rows are pulled straight out of the fused projection's [B*N, 3*H*D] output into
//              128-byte-swizzled shared tiles (npad = ceil16(N) rows each).
//   tcgen05  : S = Q K^T (128 query rows x npad keys per instruction group, both operands K-major from smem) lands
//              in tensor memory; the softmax warps read their own row (thread = TMEM lane = query), write the
//              probabilities back into TMEM as packed bf16 ON TOP of the scores they replace, and
//              O = P V runs with A = P from TMEM and B = V from smem as an MN-major operand -- V is used exactly as
//              it lies in memory ([key][d]), nothing is transposed and P never touches shared memory.
//   epilogue : O / l, bf16 (hi, lo) pair + base-2 log-sum-exp, one full 128-byte line per thread and tensor.
//
// TMEM columns (256 per CTA): scores [0, npad), probabilities [0, npad/2), output accumulator [192, 256).
#include "gemm_sm100.h"
#include "kernels.h"
#include "ptx.cuh"

#include <math_constants.h>
#include <stdlib.h>

namespace cara {
namespace {

constexpr int TC_THREADS = 160;          // warps 0-3: softmax / epilogue (TMEM lane quarter = warp), warp 4: TMA + MMA
constexpr int TC_TMEM_COLS = 256;
constexpr int TC_O_COL = 192;
constexpr int TC_D = 64;

__global__ void __launch_bounds__(TC_THREADS, 2)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_qkv, const AttnArgs a, const int npad) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t tile0 = (raw + 1023u) & ~1023u;
  const uint32_t tile_bytes = static_cast<uint32_t>(npad) * 128u;
  const uint32_t sQ = tile0, sK = tile0 + tile_bytes, sV = tile0 + 2u * tile_bytes;
  // barriers live behind the larger of (three tiles) and (Q base + 256 rows): the second query tile's MMA reads
  // 128 rows starting at row 128 whatever npad is
  const uint32_t span = 3u * tile_bytes > 32768u ? 3u * tile_bytes : 32768u;
  const uint32_t bars = tile0 + span;
  const uint32_t bar_qk = bars, bar_v = bars + 8, bar_s = bars + 16, bar_p = bars + 24, bar_o = bars + 32,
                 bar_od = bars + 40, tmem_slot = bars + 48;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int N = a.N, C = a.H * TC_D;
  const int mtiles = (N + 127) / 128;

  if (warp == 4) {
    if (lane == 0) {
      tma_prefetch_desc(&map_qkv);
      mbar_init(bar_qk, 1);
      mbar_init(bar_v, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_p, 128);
      mbar_init(bar_o, 1);
      mbar_init(bar_od, 128);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc<TC_TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();                                                  // nothing above touches global memory
  pdl_trigger();

  if (warp == 4) {
    if (lane == 0) {
      const int row0 = b * N;
      mbar_expect_tx(bar_qk, 2u * tile_bytes);
      tma_load_2d(sQ, &map_qkv, bar_qk, h * TC_D, row0);
      tma_load_2d(sK, &map_qkv, bar_qk, C + h * TC_D, row0);
      mbar_expect_tx(bar_v, tile_bytes);
      tma_load_2d(sV, &map_qkv, bar_v, 2 * C + h * TC_D, row0);
      const uint32_t idesc_s = umma_idesc_bf16_major(128, npad, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16_major(128, TC_D, 0, 1);
      mbar_wait(bar_qk, 0);
      for (int i = 0; i < mtiles; ++i) {
        if (i > 0) mbar_wait(bar_od, static_cast<uint32_t>(i - 1) & 1u);   // previous O has been read out of TMEM
        tc_fence_after();
        const uint64_t dq = umma_desc_sw128(sQ + static_cast<uint32_t>(i) * 16384u);
        const uint64_t dk = umma_desc_sw128(sK);
#pragma unroll
        for (int k = 0; k < TC_D / 16; ++k) umma_bf16(tmem_base, dq + 2u * k, dk + 2u * k, idesc_s, k != 0 ? 1u : 0u);
        umma_commit(bar_s);
        mbar_wait(bar_p, static_cast<uint32_t>(i) & 1u);                    // probabilities are in TMEM
        tc_fence_after();
        if (i == 0) mbar_wait(bar_v, 0);
        for (int k = 0; k < npad / 16; ++k) {
          const uint64_t dv = umma_desc_mn_sw128(sV + static_cast<uint32_t>(k) * 2048u, tile_bytes, 1024u);
          umma_bf16_ts(tmem_base + TC_O_COL, tmem_base + 8u * k, dv, idesc_o, k != 0 ? 1u : 0u);
        }
        umma_commit(bar_o);
      }
    }
  } else {
    const int t = warp * 32 + lane;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    const float sl2 = a.scale * 1.4426950408889634f;
    for (int i = 0; i < mtiles; ++i) {
      const int row = i * 128 + t;
      const bool warp_live = i * 128 + warp * 32 < N;          // warp-uniform: any valid query row in this warp
      mbar_wait(bar_s, static_cast<uint32_t>(i) & 1u);
      tc_fence_after();
      float mx = -CUDART_INF_F, l = 0.f;
      if (warp_live) {
        // pass 1: row maximum over the valid keys
        int c0 = 0;
        for (; c0 + 32 <= npad; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(lane_addr + c0, r);
          tmem_ld_wait();
          if (c0 + 32 <= N) {
#pragma unroll
            for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(r[j]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (c0 + j < N) mx = fmaxf(mx, __uint_as_float(r[j]));
          }
        }
        if (c0 < npad) {
          uint32_t r[16];
          tmem_ld16(lane_addr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) if (c0 + j < N) mx = fmaxf(mx, __uint_as_float(r[j]));
        }
        // pass 2: p = 2^(s*sl2 - max*sl2), row sum, packed bf16 back into TMEM (column c/2 <- keys c, c+1).
        // Chunk c0 of P overwrites score columns [c0/2, c0/2+16) which this thread has already consumed.
        const float msc = mx * sl2;
        for (c0 = 0; c0 + 32 <= npad; c0 += 32) {
          uint32_t r[32], pk[16];
          tmem_ld32(lane_addr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float p0 = exp2f(fmaf(__uint_as_float(r[2 * j]), sl2, -msc));
            float p1 = exp2f(fmaf(__uint_as_float(r[2 * j + 1]), sl2, -msc));
            if (c0 + 2 * j >= N) p0 = 0.f;
            if (c0 + 2 * j + 1 >= N) p1 = 0.f;
            l += p0 + p1;
            pk[j] = pack_bf16(p0, p1);
          }
          tmem_st16(lane_addr + (c0 >> 1), pk);
        }
        if (c0 < npad) {
          uint32_t r[16], pk[8];
          tmem_ld16(lane_addr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float p0 = exp2f(fmaf(__uint_as_float(r[2 * j]), sl2, -msc));
            float p1 = exp2f(fmaf(__uint_as_float(r[2 * j + 1]), sl2, -msc));
            if (c0 + 2 * j >= N) p0 = 0.f;
            if (c0 + 2 * j + 1 >= N) p1 = 0.f;
            l += p0 + p1;
            pk[j] = pack_bf16(p0, p1);
          }
          tmem_st8(lane_addr + (c0 >> 1), pk);
        }
        tmem_st_wait();
      }
      tc_fence_before();
      mbar_arrive(bar_p);
      mbar_wait(bar_o, static_cast<uint32_t>(i) & 1u);
      tc_fence_after();
      uint32_t o[64];
      if (warp_live) {
        tmem_ld32(lane_addr + TC_O_COL, *reinterpret_cast<uint32_t(*)[32]>(&o[0]));
        tmem_ld32(lane_addr + TC_O_COL + 32, *reinterpret_cast<uint32_t(*)[32]>(&o[32]));
        tmem_ld_wait();
      }
      tc_fence_before();
      mbar_arrive(bar_od);
      if (warp_live && row < N) {
        const float inv = 1.0f / l;
        const long off = (static_cast<long>(b) * N + row) * C + h * TC_D;
        __nv_bfloat16* po = a.o + off;
        __nv_bfloat16* pl = a.o_lo != nullptr ? a.o_lo + off : nullptr;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float v[16];
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int e = 0; e < 16; ++e) v[e] = __uint_as_float(o[16 * j + e]) * inv;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            hi[e] = pack_bf16(v[2 * e], v[2 * e + 1]);
            const float2 hf = unpack_bf16(hi[e]);
            lo[e] = pack_bf16(v[2 * e] - hf.x, v[2 * e + 1] - hf.y);
          }
          st_global_v8(po + 16 * j, hi);
          if (pl != nullptr) st_global_v8(pl + 16 * j, lo);
        }
        if (a.lse != nullptr) a.lse[(static_cast<long>(b) * a.H + h) * N + row] = mx * sl2 + log2f(l);
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc<TC_TMEM_COLS>(tmem_base);
  }
}


// [r2b] The same forward with EIGHT softmax warps: two per TMEM lane quarter, each taking half of the key columns of its
// query row.  The softmax (two passes over the row in tensor memory + the exp) is the serial part of a head -- with four
// warps the CTA spends most of its time there while the tensor pipe waits -- so halving it shortens every tile.
//   * half 0 owns score columns [0, split), half 1 [split, npad); each packs its probabilities over its OWN consumed
//     scores ([0, split/2) and [split, split + (npad - split)/2)), so the halves never touch each other's columns and
//     the P V MMA reads k-step j from column (16j < split ? 8j : split + (16j - split)/2);
//   * the two partial row maxima (and later the two partial row sums) cross through shared memory with one 64-thread
//     named barrier per lane quarter;
//   * the epilogue splits the 64 output columns the same way (32 per thread).
constexpr int TC8_THREADS = 288;         // warps 0-7: softmax / epilogue (lane quarter = warp & 3, column half = warp >> 2), warp 8: TMA + MMA

// one named barrier per lane quarter (immediate ids, so ptxas reserves 5 barriers per CTA and not all 16)
__device__ __forceinline__ void pair_sync(int q4) {
  switch (q4) {
    case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
    case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
    case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
    default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
  }
}

__global__ void __launch_bounds__(TC8_THREADS, 2)
attn_fwd_tc8_kernel(const __grid_constant__ CUtensorMap map_qkv, const AttnArgs a, const int npad) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t tile0 = (raw + 1023u) & ~1023u;
  const uint32_t tile_bytes = static_cast<uint32_t>(npad) * 128u;
  const uint32_t sQ = tile0, sK = tile0 + tile_bytes, sV = tile0 + 2u * tile_bytes;
  const uint32_t span = 3u * tile_bytes > 32768u ? 3u * tile_bytes : 32768u;
  const uint32_t bars = tile0 + span;
  const uint32_t bar_qk = bars, bar_v = bars + 8, bar_s = bars + 16, bar_p = bars + 24, bar_o = bars + 32,
                 bar_od = bars + 40, tmem_slot = bars + 48, xch = bars + 64;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));
  float* s_max = reinterpret_cast<float*>(smem_raw + (xch - raw));       // [2 halves][128 rows]
  float* s_sum = s_max + 256;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N, C = a.H * TC_D;
  const int mtiles = (N + 127) / 128;
  const int split = ((npad / 16 + 1) / 2) * 16;
  const int heads = a.B * a.H;                                 // persistent: this CTA takes heads blockIdx.x, + gridDim.x, ...

  if (warp == 8) {
    if (lane == 0) {
      tma_prefetch_desc(&map_qkv);
      mbar_init(bar_qk, 1);
      mbar_init(bar_v, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_p, 256);
      mbar_init(bar_o, 1);
      mbar_init(bar_od, 256);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc<TC_TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();
  pdl_trigger();

  if (warp == 8) {
    if (lane == 0) {
      // The next head's Q / K are requested the moment this head's last S = Q K^T has retired, its V the moment the
      // last P V has retired: with two resident CTAs per SM and 78 KB per head, a CTA that only starts loading when it
      // starts a head leaves the memory system with too little in flight (2.7 TB/s).
      auto load_qk = [&](int head) {
        const int row0 = (head / a.H) * N, col = (head % a.H) * TC_D;
        mbar_expect_tx(bar_qk, 2u * tile_bytes);
        tma_load_2d(sQ, &map_qkv, bar_qk, col, row0);
        tma_load_2d(sK, &map_qkv, bar_qk, C + col, row0);
      };
      auto load_v = [&](int head) {
        const int row0 = (head / a.H) * N, col = (head % a.H) * TC_D;
        mbar_expect_tx(bar_v, tile_bytes);
        tma_load_2d(sV, &map_qkv, bar_v, 2 * C + col, row0);
      };
      const uint32_t idesc_s = umma_idesc_bf16_major(128, npad, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16_major(128, TC_D, 0, 1);
      uint32_t it = 0, n = 0;
      if (static_cast<int>(blockIdx.x) < heads) {
        load_qk(blockIdx.x);
        load_v(blockIdx.x);
      }
      for (int head = blockIdx.x; head < heads; head += gridDim.x, ++it) {
        const int next = head + static_cast<int>(gridDim.x);
        mbar_wait(bar_qk, it & 1u);
        for (int i = 0; i < mtiles; ++i, ++n) {
          if (n > 0) mbar_wait(bar_od, (n - 1u) & 1u);                       // previous O has been read out of TMEM
          tc_fence_after();
          const uint64_t dq = umma_desc_sw128(sQ + static_cast<uint32_t>(i) * 16384u);
          const uint64_t dk = umma_desc_sw128(sK);
#pragma unroll
          for (int k = 0; k < TC_D / 16; ++k) umma_bf16(tmem_base, dq + 2u * k, dk + 2u * k, idesc_s, k != 0 ? 1u : 0u);
          umma_commit(bar_s);
          if (i == mtiles - 1 && next < heads) {                             // Q / K are dead once the last S has retired
            mbar_wait(bar_s, n & 1u);
            load_qk(next);
          }
          mbar_wait(bar_p, n & 1u);                                          // probabilities are in TMEM
          tc_fence_after();
          if (i == 0) mbar_wait(bar_v, it & 1u);
          for (int k = 0; k < npad / 16; ++k) {
            const int c = 16 * k;
            const uint32_t pcol = static_cast<uint32_t>(c < split ? (c >> 1) : split + ((c - split) >> 1));
            const uint64_t dv = umma_desc_mn_sw128(sV + static_cast<uint32_t>(k) * 2048u, tile_bytes, 1024u);
            umma_bf16_ts(tmem_base + TC_O_COL, tmem_base + pcol, dv, idesc_o, k != 0 ? 1u : 0u);
          }
          umma_commit(bar_o);
          if (i == mtiles - 1 && next < heads) {                             // V is dead once the last P V has retired
            mbar_wait(bar_o, n & 1u);
            load_v(next);
          }
        }
      }
    }
  } else {
    const int q4 = warp & 3, half = warp >> 2;
    const int t = q4 * 32 + lane;                                  // query row of this thread inside the tile
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const float sl2 = a.scale * 1.4426950408889634f;
    const int cb = half == 0 ? 0 : split, ce = half == 0 ? split : npad;
    uint32_t n = 0;
    for (int head = blockIdx.x; head < heads; head += gridDim.x) {
    const int b = head / a.H, h = head % a.H;
    for (int i = 0; i < mtiles; ++i, ++n) {
      const int row = i * 128 + t;
      const bool warp_live = i * 128 + q4 * 32 < N;               // uniform over the two warps of a lane quarter
      mbar_wait(bar_s, n & 1u);
      tc_fence_after();
      float mx = -CUDART_INF_F, l = 0.f;
      if (warp_live) {
        // pass 1: maximum over this half's valid keys, then the row maximum through shared memory
        int c0 = cb;
        for (; c0 + 32 <= ce; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(lane_addr + c0, r);
          tmem_ld_wait();
          if (c0 + 32 <= N) {
#pragma unroll
            for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(r[j]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (c0 + j < N) mx = fmaxf(mx, __uint_as_float(r[j]));
          }
        }
        if (c0 < ce) {
          uint32_t r[16];
          tmem_ld16(lane_addr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) if (c0 + j < N) mx = fmaxf(mx, __uint_as_float(r[j]));
        }
        s_max[half * 128 + t] = mx;
        pair_sync(q4);
        mx = fmaxf(mx, s_max[(half ^ 1) * 128 + t]);               // (half 0 always holds a valid key: finite)
        // pass 2: p = 2^(s*sl2 - max*sl2), partial row sum, packed bf16 over this half's own consumed scores
        const float msc = mx * sl2;
        for (c0 = cb; c0 + 32 <= ce; c0 += 32) {
          uint32_t r[32], pk[16];
          tmem_ld32(lane_addr + c0, r);
          tmem_ld_wait();
          if (c0 + 32 <= N) {                                      // (only the chunk that straddles N pays for the mask)
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float p0 = exp2f(fmaf(__uint_as_float(r[2 * j]), sl2, -msc));
              const float p1 = exp2f(fmaf(__uint_as_float(r[2 * j + 1]), sl2, -msc));
              l += p0 + p1;
              pk[j] = pack_bf16(p0, p1);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float p0 = exp2f(fmaf(__uint_as_float(r[2 * j]), sl2, -msc));
              float p1 = exp2f(fmaf(__uint_as_float(r[2 * j + 1]), sl2, -msc));
              if (c0 + 2 * j >= N) p0 = 0.f;
              if (c0 + 2 * j + 1 >= N) p1 = 0.f;
              l += p0 + p1;
              pk[j] = pack_bf16(p0, p1);
            }
          }
          tmem_st16(lane_addr + cb + ((c0 - cb) >> 1), pk);
        }
        if (c0 < ce) {
          uint32_t r[16], pk[8];
          tmem_ld16(lane_addr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float p0 = exp2f(fmaf(__uint_as_float(r[2 * j]), sl2, -msc));
            float p1 = exp2f(fmaf(__uint_as_float(r[2 * j + 1]), sl2, -msc));
            if (c0 + 2 * j >= N) p0 = 0.f;
            if (c0 + 2 * j + 1 >= N) p1 = 0.f;
            l += p0 + p1;
            pk[j] = pack_bf16(p0, p1);
          }
          tmem_st8(lane_addr + cb + ((c0 - cb) >> 1), pk);
        }
        tmem_st_wait();
        s_sum[half * 128 + t] = l;
      }
      tc_fence_before();
      mbar_arrive(bar_p);
      mbar_wait(bar_o, n & 1u);
      tc_fence_after();
      uint32_t o[32];
      if (warp_live) {
        tmem_ld32(lane_addr + TC_O_COL + 32 * half, o);
        tmem_ld_wait();
      }
      tc_fence_before();
      mbar_arrive(bar_od);
      if (warp_live) {
        pair_sync(q4);                                             // the partner's partial sum is in shared memory
        l += s_sum[(half ^ 1) * 128 + t];
        if (row < N) {
          const float inv = 1.0f / l;
          const long off = (static_cast<long>(b) * N + row) * C + h * TC_D + 32 * half;
          __nv_bfloat16* po = a.o + off;
          __nv_bfloat16* pl = a.o_lo != nullptr ? a.o_lo + off : nullptr;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            float v[16];
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = __uint_as_float(o[16 * j + e]) * inv;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              hi[e] = pack_bf16(v[2 * e], v[2 * e + 1]);
              const float2 hf = unpack_bf16(hi[e]);
              lo[e] = pack_bf16(v[2 * e] - hf.x, v[2 * e + 1] - hf.y);
            }
            st_global_v8(po + 16 * j, hi);
            if (pl != nullptr) st_global_v8(pl + 16 * j, lo);
          }
          if (half == 0 && a.lse != nullptr) a.lse[(static_cast<long>(b) * a.H + h) * N + row] = mx * sl2 + log2f(l);
        }
      }
    }
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc<TC_TMEM_COLS>(tmem_base);
  }
}


// ------------------------------------------------------------------------------------ backward
// Pre-pass (HBM-bound, one warp per token row): delta[b,h,n] = sum_d dO[n,h,d] (O + O_lo)[n,h,d].
// O is carried as a bf16 (hi, lo) pair because with plain bf16 O the rows of dS stop summing to ~0 for peaked
// softmax rows and dq / dk lose the parity bar.
__global__ void __launch_bounds__(256)
attn_delta_kernel(const __nv_bfloat16* __restrict__ d_o, const __nv_bfloat16* __restrict__ o,
                  const __nv_bfloat16* __restrict__ o_lo, float* __restrict__ delta, int rows, int N, int H) {
  pdl_wait();
  pdl_trigger();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int b = row / N, n = row % N;
  const long base = static_cast<long>(row) * H * TC_D;
  for (int i = lane; i < H * 8; i += 32) {                       // 16-byte chunk i: head i / 8
    const uint4 x = *reinterpret_cast<const uint4*>(d_o + base + i * 8);
    const uint4 y = *reinterpret_cast<const uint4*>(o + base + i * 8);
    const uint4 z = *reinterpret_cast<const uint4*>(o_lo + base + i * 8);
    const uint32_t xw[4] = {x.x, x.y, x.z, x.w}, yw[4] = {y.x, y.y, y.z, y.w}, zw[4] = {z.x, z.y, z.z, z.w};
    float acc = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 xf = unpack_bf16(xw[e]), yf = unpack_bf16(yw[e]), zf = unpack_bf16(zw[e]);
      acc += xf.x * (yf.x + zf.x) + xf.y * (yf.y + zf.y);
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    acc += __shfl_xor_sync(0xffffffffu, acc, 4);
    if ((lane & 7) == 0) delta[(static_cast<long>(b) * H + (i >> 3)) * N + n] = acc;
  }
}

// One persistent CTA per SM walks over (sample, head) pairs.  Per head and 128-key tile t (keys on the TMEM lanes):
//   S^T  = K_t Q^T            -> TMEM [0, npad)            (both operands K-major from smem)
//   dP^T = V_t dO^T           -> TMEM [256, 256 + npad)
//   threads (lane = key, two warps per lane quarter splitting the query columns):
//        P^T  = 2^(S^T sl2 - lse[q])                 -> bf16 back into TMEM over the scores it replaces
//        dS^T = P^T (.) (dP^T - delta[q])            -> bf16 into ONE shared tile laid out [64-query block][key][128 B]
//   dV_t  = P^T dO            A = P^T from TMEM,  B = dO as it lies in memory (MN-major)          -> TMEM [256, 320)
//   dK_t  = dS^T Q            A = the shared tile read K-major,  B = Q (MN-major)                 -> TMEM [320, 384)
//   dQ   += dS K_t            A = THE SAME shared tile read MN-major (M = query), B = K_t (MN-major) -> TMEM [384, 512)
// so the [N, N] matrices never leave the SM, nothing is transposed by the SIMT cores, and the only shared-memory
// staging is the single dS^T tile.  dQ partials of the two key tiles are summed in registers.
constexpr int TCB_THREADS = 288;         // warps 0-7: compute (lane quarter = warp & 3, column half = warp >> 2); warp 8: TMA + MMA
constexpr int TCB_DS_BYTES = 65536;      // 4 query blocks x 128 keys x 128 B
constexpr int TCB_DP_COL = 256, TCB_DV_COL = 256, TCB_DK_COL = 320, TCB_DQ_COL = 384;

__device__ long long g_attn_dbg[64];
#ifdef CARA_ATTN_DEBUG
#define DBG_STAMP(i) do { if (blockIdx.x == 0 && (i) < 64) g_attn_dbg[(i)] = clock64(); } while (0)
#else
#define DBG_STAMP(i) do { } while (0)
#endif

__device__ __forceinline__ void named_bar_sync_256() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__global__ void __launch_bounds__(TCB_THREADS, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do,
                   const AttnArgs a, const int npad, const int qk_pairs) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t tile0 = (raw + 1023u) & ~1023u;
  const uint32_t tile_bytes = static_cast<uint32_t>(npad) * 128u;
  // Input tiles: qk_pairs (1 or 2) x {Q, K}, then V, dO.  With two Q/K pairs (whenever they fit: N <= 208) the next
  // head's Q and K land while this head is being computed; V / dO are reloaded in place as soon as the last MMA
  // that reads them has retired (V: last dP^T, dO: last dV), so no load is exposed between heads.
  // The second key tile's A operands read 128 rows from row 128 of K / V whatever npad is: what lies behind them
  // (the next tile, then the dS^T tile) is allocated and always holds finite bf16 data (possibly mid-reload).
  const uint32_t sV = tile0 + 2u * static_cast<uint32_t>(qk_pairs) * tile_bytes, sDO = sV + tile_bytes;
  const uint32_t sDS = sDO + tile_bytes;
  const uint32_t stats = sDS + TCB_DS_BYTES;                 // nlse[256], delta[256] (fp32)
  const uint32_t bars = stats + 2048u;
  const uint32_t bar_sdp = bars + 8, bar_pds = bars + 16, bar_kv = bars + 24, bar_out = bars + 32,
                 bar_rd = bars + 40, tmem_slot = bars + 48, bar_qk0 = bars + 56, bar_v = bars + 72, bar_do = bars + 80,
                 bar_pds0 = bars + 88;
  float* s_nlse = reinterpret_cast<float*>(smem_raw + (stats - raw));
  float* s_delta = s_nlse + 256;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N, C = a.H * TC_D;
  const int nt = (N + 127) / 128;                              // key tiles == query tiles
  const int ksteps = npad / 16;
  // The query columns are worked through in two phases so that the dV / dK MMAs over the first 128 queries run
  // while the compute warps are still busy with the rest: phase 0 = queries [0, qa), phase 1 = [128, npad); in each
  // phase compute half 0 takes the lower part and half 1 the upper part.  Every (phase, half) segment
  // [sb, se) packs its P^T into TMEM columns [sb, sb + (se - sb) / 2) -- inside its own, already consumed, scores.
  const int qa = npad < 128 ? npad : 128;
  const int a_split = ((qa / 16 + 1) / 2) * 16;
  const int r_split = 128 + (((npad - qa) / 16 + 1) / 2) * 16;
  const int heads = a.B * a.H;

  if (warp == 8) {
    if (lane == 0) {
      tma_prefetch_desc(&map_qkv);
      tma_prefetch_desc(&map_do);
      mbar_init(bar_qk0, 1);
      mbar_init(bar_qk0 + 8, 1);
      mbar_init(bar_v, 1);
      mbar_init(bar_do, 1);
      mbar_init(bar_sdp, 1);
      mbar_init(bar_pds, 256);
      mbar_init(bar_pds0, 256);
      mbar_init(bar_kv, 1);
      mbar_init(bar_out, 1);
      mbar_init(bar_rd, 256);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc<512>(tmem_slot);
  } else {
    // the dS^T tile may be read (as don't-care rows / columns) before it is ever written: make it finite
    for (uint32_t off = threadIdx.x * 16u; off < TCB_DS_BYTES; off += 256u * 16u)
      asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(sDS + off), "r"(0u) : "memory");
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  pdl_wait();                                                  // nothing above touches global memory
  pdl_trigger();

  if (warp == 8) {
    if (lane == 0) {
      auto head_coords = [&](int head, int& row0, int& col) { row0 = (head / a.H) * N; col = (head % a.H) * TC_D; };
      auto load_qk = [&](int head, uint32_t pair) {
        int row0, col;
        head_coords(head, row0, col);
        const uint32_t q = tile0 + 2u * pair * tile_bytes, bar = bar_qk0 + 8u * pair;
        mbar_expect_tx(bar, 2u * tile_bytes);
        tma_load_2d(q + tile_bytes, &map_qkv, bar, C + col, row0);
        tma_load_2d(q, &map_qkv, bar, col, row0);
      };
      auto load_v = [&](int head) {
        int row0, col;
        head_coords(head, row0, col);
        mbar_expect_tx(bar_v, tile_bytes);
        tma_load_2d(sV, &map_qkv, bar_v, 2 * C + col, row0);
      };
      auto load_do = [&](int head) {
        int row0, col;
        head_coords(head, row0, col);
        mbar_expect_tx(bar_do, tile_bytes);
        tma_load_2d(sDO, &map_do, bar_do, col, row0);
      };
      const uint32_t idesc_s = umma_idesc_bf16_major(128, npad, 0, 0);
      constexpr uint32_t idesc_dv = umma_idesc_bf16_major(128, TC_D, 0, 1);   // A from TMEM (K-major), B MN-major
      constexpr uint32_t idesc_dk = umma_idesc_bf16_major(128, TC_D, 0, 1);   // A K-major smem, B MN-major
      constexpr uint32_t idesc_dq = umma_idesc_bf16_major(128, TC_D, 1, 1);   // A MN-major smem, B MN-major
      uint32_t it = 0, n = 0;
      if (static_cast<int>(blockIdx.x) < heads) {
        load_qk(blockIdx.x, 0);
        load_v(blockIdx.x);
        load_do(blockIdx.x);
      }
      for (int head = blockIdx.x; head < heads; head += gridDim.x, ++it) {
        const int next = head + static_cast<int>(gridDim.x);
        const uint32_t pair = qk_pairs == 2 ? (it & 1u) : 0u;
        const uint32_t sQ = tile0 + 2u * pair * tile_bytes, sK = sQ + tile_bytes;
        // the other Q/K pair was last read by the previous head, whose MMAs have all retired (wait at its end)
        if (qk_pairs == 2 && next < heads) load_qk(next, pair ^ 1u);
        mbar_wait(bar_qk0 + 8u * pair, (qk_pairs == 2 ? (it >> 1) : it) & 1u);
        if (it == 1) DBG_STAMP(0);
        for (int t = 0; t < nt; ++t, ++n) {
          if (n > 0) mbar_wait(bar_rd, (n - 1u) & 1u);         // previous outputs have been read out of TMEM
          tc_fence_after();
          if (it == 1) DBG_STAMP(1 + 8 * t);
          {
            const uint64_t dk = umma_desc_sw128(sK + static_cast<uint32_t>(t) * 16384u), dq = umma_desc_sw128(sQ);
#pragma unroll
            for (int k = 0; k < TC_D / 16; ++k) umma_bf16(tmem_base, dk + 2u * k, dq + 2u * k, idesc_s, k != 0 ? 1u : 0u);
            if (t == 0) {
              mbar_wait(bar_v, it & 1u);
              mbar_wait(bar_do, it & 1u);
              tc_fence_after();
            }
            const uint64_t dv = umma_desc_sw128(sV + static_cast<uint32_t>(t) * 16384u), dd = umma_desc_sw128(sDO);
#pragma unroll
            for (int k = 0; k < TC_D / 16; ++k)
              umma_bf16(tmem_base + TCB_DP_COL, dv + 2u * k, dd + 2u * k, idesc_s, k != 0 ? 1u : 0u);
          }
          umma_commit(bar_sdp);
          if (t == nt - 1 && next < heads) {                    // V is dead once the last dP^T has retired
            mbar_wait(bar_sdp, n & 1u);
            load_v(next);
          }
          // dV_t = P^T dO,  dK_t = dS^T Q   (K = queries): the k-steps of phase 0 start as soon as both compute
          // halves are done with the first 128 queries (whose dP^T columns the two accumulators overlay)
          auto dv_dk = [&](int j) {
            const int c = 16 * j;
            const int sb = c < a_split ? 0 : (c < qa ? a_split : (c < r_split ? 128 : r_split));
            umma_bf16_ts(tmem_base + TCB_DV_COL, tmem_base + static_cast<uint32_t>(sb + ((c - sb) >> 1)),
                         umma_desc_mn_sw128(sDO + static_cast<uint32_t>(j) * 2048u, tile_bytes, 1024u), idesc_dv,
                         j != 0 ? 1u : 0u);
            umma_bf16(tmem_base + TCB_DK_COL,
                      umma_desc_sw128(sDS + static_cast<uint32_t>(j >> 2) * 16384u + static_cast<uint32_t>(j & 3) * 32u),
                      umma_desc_mn_sw128(sQ + static_cast<uint32_t>(j) * 2048u, tile_bytes, 1024u), idesc_dk,
                      j != 0 ? 1u : 0u);
          };
          mbar_wait(bar_pds0, n & 1u);                          // P^T / dS^T of queries [0, qa) are in place
          tc_fence_after();
          for (int j = 0; j < qa / 16; ++j) dv_dk(j);
          mbar_wait(bar_pds, n & 1u);                           // ... and the rest
          tc_fence_after();
          if (it == 1) DBG_STAMP(2 + 8 * t);
          for (int j = qa / 16; j < ksteps; ++j) dv_dk(j);
          umma_commit(bar_kv);                                  // dK_t / dV_t can be read out while dQ still runs
          const int kk = (npad - 128 * t < 128 ? npad - 128 * t : 128) / 16;   // valid keys of this tile / 16
          for (int j = 0; j < kk; ++j) {                        // dQ_m = dS K_t   (K = keys of tile t), m interleaved
            for (int m = 0; m < nt; ++m) {
              umma_bf16(tmem_base + TCB_DQ_COL + 64u * m,
                        umma_desc_mn_sw128(sDS + static_cast<uint32_t>(2 * m) * 16384u + static_cast<uint32_t>(j) * 2048u,
                                           16384u, 1024u),
                        umma_desc_mn_sw128(sK + static_cast<uint32_t>(t) * 16384u + static_cast<uint32_t>(j) * 2048u,
                                           tile_bytes, 1024u),
                        idesc_dq, j != 0 ? 1u : 0u);
            }
          }
          umma_commit(bar_out);
          if (t == nt - 1 && next < heads) {                    // dO is dead once the last dV has retired
            mbar_wait(bar_kv, n & 1u);
            load_do(next);
          }
          if (it == 1) DBG_STAMP(3 + 8 * t);
        }
        // every MMA that reads this head's Q / K has been issued; once they retire that pair may be refilled
        mbar_wait(bar_out, (n - 1u) & 1u);
        if (it == 1) DBG_STAMP(20);
        if (qk_pairs == 1 && next < heads) load_qk(next, 0);
      }
    }
  } else {
    const int q4 = warp & 3, half = warp >> 2;
    const int tid = threadIdx.x;                                // 0..255
    const int key_local = q4 * 32 + lane;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q4 * 32) << 16);
    const float sl2 = a.scale * 1.4426950408889634f;
    const uint32_t ds_row = sDS + static_cast<uint32_t>(key_local) * 128u;
    const uint32_t sw = static_cast<uint32_t>(key_local & 7);
    uint32_t n = 0, it = 0;
    for (int head = blockIdx.x; head < heads; head += gridDim.x, ++it) {
      const int b = head / a.H, h = head % a.H;
      // ---- per-head statistics (everyone is past the previous head's last use of them: see bar_pds / bar_out)
      {
        const long sb = (static_cast<long>(b) * a.H + h) * N;
        s_nlse[tid] = tid < N ? -a.lse[sb + tid] : -1e30f;
        s_delta[tid] = tid < N ? a.delta[sb + tid] : 0.f;
        named_bar_sync_256();
      }
      if (it == 1 && tid == 0) DBG_STAMP(32);
      float dq[64];
#pragma unroll
      for (int j = 0; j < 64; ++j) dq[j] = 0.f;
      __nv_bfloat16* gbase = a.dqkv + static_cast<long>(b) * N * 3 * C + h * TC_D;

      for (int t = 0; t < nt; ++t, ++n) {
        const int key = t * 128 + key_local;
        const bool key_ok = key < N;
        const bool warp_live = t * 128 + q4 * 32 < npad;        // warp-uniform
        mbar_wait(bar_sdp, n & 1u);
        tc_fence_after();
        if (it == 1 && tid == 0) DBG_STAMP(33 + 8 * t);
        // one (phase, half) segment [cb, ce) of the query columns, P^T packed from column cb on
        auto segment = [&](int cb, int ce) {
          for (int c = cb; c < ce; c += 16) {
            uint32_t s[16], dp[16], pk[8], dsk[8];
            tmem_ld16(lane_addr + c, s);
            tmem_ld16(lane_addr + TCB_DP_COL + c, dp);
            tmem_ld_wait();
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 L = *reinterpret_cast<const float4*>(s_nlse + c + 4 * j4);
              const float4 Dl = *reinterpret_cast<const float4*>(s_delta + c + 4 * j4);
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
            // P^T: 16 queries of this key -> 8 packed columns on top of already consumed scores
            tmem_st8(lane_addr + static_cast<uint32_t>(cb + ((c - cb) >> 1)), pk);
            // dS^T: two 16-byte chunks of row `key_local` in query block c / 64
            const uint32_t blk = ds_row + static_cast<uint32_t>(c >> 6) * 16384u;
            const uint32_t ch = static_cast<uint32_t>((c & 63) >> 3);
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(blk + ((ch ^ sw) << 4)), "r"(dsk[0]), "r"(dsk[1]),
                         "r"(dsk[2]), "r"(dsk[3]) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(blk + (((ch + 1u) ^ sw) << 4)), "r"(dsk[4]),
                         "r"(dsk[5]), "r"(dsk[6]), "r"(dsk[7]) : "memory");
          }
          // keys in [N, npad) are padding: their rows of dS^T feed dQ and must be exactly zero (their scores are
          // finite garbage -- the next sample's rows -- so the values written above may be anything, even inf/nan)
          if (!key_ok) {
            for (int c = cb; c < ce; c += 8) {
              const uint32_t blk = ds_row + static_cast<uint32_t>(c >> 6) * 16384u;
              const uint32_t ch = static_cast<uint32_t>((c & 63) >> 3);
              asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(blk + ((ch ^ sw) << 4)), "r"(0u) : "memory");
            }
          }
          tmem_st_wait();
          fence_proxy_async();                                  // dS^T stores -> visible to the tensor core (async proxy)
        };
        if (warp_live) segment(half == 0 ? 0 : a_split, half == 0 ? a_split : qa);
        tc_fence_before();
        mbar_arrive(bar_pds0);
        if (warp_live) segment(half == 0 ? 128 : r_split, half == 0 ? r_split : npad);
        tc_fence_before();
        mbar_arrive(bar_pds);
        if (it == 1 && tid == 0) DBG_STAMP(34 + 8 * t);
        // ---- read out: half 0 -> dK_t rows, half 1 -> dV_t rows (while the dQ MMAs are still running)
        mbar_wait(bar_kv, n & 1u);
        tc_fence_after();
        if (it == 1 && tid == 0) DBG_STAMP(35 + 8 * t);
        if (warp_live) {
          const uint32_t col = half == 0 ? TCB_DK_COL : TCB_DV_COL;
          const float sc = half == 0 ? a.scale : 1.0f;
          __nv_bfloat16* dst = gbase + static_cast<long>(key) * 3 * C + (half == 0 ? C : 2 * C);
#pragma unroll
          for (int part = 0; part < 2; ++part) {
            uint32_t r[32];
            tmem_ld32(lane_addr + col + 32 * part, r);
            tmem_ld_wait();
            if (key_ok) {
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
        }
        // ---- dQ partial of query tile `half` (lane = query) accumulated over the key tiles in registers
        mbar_wait(bar_out, n & 1u);
        tc_fence_after();
        if (it == 1 && tid == 0) DBG_STAMP(36 + 8 * t);
        if (half < nt) {
#pragma unroll
          for (int part = 0; part < 2; ++part) {
            uint32_t r[32];
            tmem_ld32(lane_addr + TCB_DQ_COL + 64 * half + 32 * part, r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) dq[32 * part + j] += __uint_as_float(r[j]);
          }
        }
        tc_fence_before();
        mbar_arrive(bar_rd);
        if (it == 1 && tid == 0) DBG_STAMP(37 + 8 * t);
      }
      // ---- dQ rows of query tile `half`
      const int qrow = half * 128 + key_local;
      if (half < nt && qrow < N) {
        __nv_bfloat16* dst = gbase + static_cast<long>(qrow) * 3 * C;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t w[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) w[e] = pack_bf16(dq[16 * j + 2 * e] * a.scale, dq[16 * j + 2 * e + 1] * a.scale);
          st_global_v8(dst + 16 * j, w);
        }
      }
      if (it == 1 && tid == 0) DBG_STAMP(60);
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

}  // namespace

// D = 64, N <= 256: tcgen05 path.  Returns 1 when the shape is not covered (caller falls back to the mma.sync kernel).
int attn_fwd_tc_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.D != TC_D || a.N > 256 || a.N < 1) return 1;
  const int npad = ((a.N + 15) / 16) * 16;
  const long rows = static_cast<long>(a.B) * a.N;
  const long cols = 3L * a.H * TC_D;
  CUtensorMap map;
  if (make_map_bf16(&map, a.qkv, rows, cols, cols, npad) != 0) return -54;
  const int tile_bytes = npad * 128;
  const int span = 3 * tile_bytes > 32768 ? 3 * tile_bytes : 32768;
  const int smem = 1024 + span + 64;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(attn_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 1024 + 3 * 256 * 128 + 64) !=
        cudaSuccess)
      return -52;
    configured = true;
  }
  // [r2b] eight softmax warps (CARA_ATTN_FWD8=0: the four-warp kernel)
  static int fwd8 = -1;
  if (fwd8 < 0) { const char* e = getenv("CARA_ATTN_FWD8"); fwd8 = e != nullptr ? atoi(e) : 1; }
  if (fwd8) {
    static bool configured8 = false;
    if (!configured8) {
      if (cudaFuncSetAttribute(attn_fwd_tc8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               1024 + 3 * 256 * 128 + 64 + 2048) != cudaSuccess)
        return -52;
      configured8 = true;
    }
    // persistent: two resident CTAs per SM walk over the (sample, head) pairs (CARA_ATTN_FWD8=2: one CTA per pair)
    static int sms = 0;
    if (sms == 0) {
      int dev = 0;
      if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    int grid = a.B * a.H;
    if (fwd8 == 1 && grid > 2 * sms) grid = 2 * sms;
    return launch_pdl_f<2>(attn_fwd_tc8_kernel, dim3(grid), dim3(TC8_THREADS), smem + 2048, st, map, a, npad) == cudaSuccess ? 0 : -53;
  }
  return launch_pdl_f<2>(attn_fwd_tc_kernel, dim3(a.B * a.H), dim3(TC_THREADS), smem, st, map, a, npad) == cudaSuccess ? 0 : -53;
}

}  // namespace cara

namespace cara {
int attn_bwd_tc_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.D != TC_D || a.N > 256 || a.N < 1 || a.delta == nullptr) return 1;
  const int npad = ((a.N + 15) / 16) * 16;
  const long rows = static_cast<long>(a.B) * a.N;
  const long C = static_cast<long>(a.H) * TC_D;
  CUtensorMap map_qkv, map_do;
  if (make_map_bf16(&map_qkv, a.qkv, rows, 3 * C, 3 * C, npad) != 0) return -54;
  if (make_map_bf16(&map_do, a.d_o, rows, C, C, npad) != 0) return -54;
  int qk_pairs = 2;                                             // prefetch the next head's Q / K when they fit
  int smem = 1024 + 6 * npad * 128 + TCB_DS_BYTES + 2048 + 128;
  if (smem > 232448) {
    qk_pairs = 1;
    smem = 1024 + 4 * npad * 128 + TCB_DS_BYTES + 2048 + 128;
  }
  static int configured = 0;
  if (configured < smem) {
    if (cudaFuncSetAttribute(attn_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -52;
    configured = smem;
  }
  int grid = a.B * a.H;
  if (grid > 148) grid = 148;
  // a.o == nullptr: delta was written by the output projection's dX GEMM (EPI_DELTA), no pre-pass
  if (a.o != nullptr &&
      launch_pdl_f<2>(attn_delta_kernel, dim3(static_cast<int>((rows + 7) / 8)), dim3(256), 0, st, a.d_o, a.o, a.o_lo, a.delta,
                 static_cast<int>(rows), a.N, a.H) != cudaSuccess)
    return -53;
  return launch_pdl_f<2>(attn_bwd_tc_kernel, dim3(grid), dim3(TCB_THREADS), smem, st, map_qkv, map_do, a, npad, qk_pairs) ==
                 cudaSuccess ? 0 : -53;
}
// rowsum(dO (.) (O + O_lo)) into a.delta: the pre-pass of the long-sequence backward (attention_long.cu)
int attn_delta_launch(const AttnArgs& a, cudaStream_t st) {
  const long rows = static_cast<long>(a.B) * a.N;
  return launch_pdl_f<2>(attn_delta_kernel, dim3(static_cast<int>((rows + 7) / 8)), dim3(256), 0, st, a.d_o, a.o, a.o_lo,
                         a.delta, static_cast<int>(rows), a.N, a.H) == cudaSuccess ? 0 : -53;
}
int attn_debug_read(long long* out, int n) {
  if (n > 64) n = 64;
  if (n <= 0 || cudaMemcpyFromSymbol(out, g_attn_dbg, sizeof(long long) * n) != cudaSuccess) return 0;
  return n;
}
}  // namespace cara
