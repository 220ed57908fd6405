// Key-tiled attention core for head size 80 (ViT-H/14) at any sequence length.  The whole-head kernels of attention.cu
// keep all of a head's K/V (and Q/dO in the backward) in shared memory, which stops at N = 432 (forward) and N = 320
// (backward).  These kernels hold only a tile of 128 (forward) or 64 (backward) rows of the operand a CTA owns, and
// stream the other operand through a 2-stage cp.async ring of 64-row windows, so shared memory does not grow with N.
//
// Every warp runs exactly the whole-head kernel's sequence of chunk calls (attention_mma.cuh): full 64-row chunks, then
// the same remainder of 1-3 16-row steps, at the same absolute row indices.  The inputs each call sees are the same
// (rows >= N are zero in both), so wherever both paths run, o, o_lo, lse and dqkv are bit-identical to theirs.
//
//   attn_fwd_tiled_kernel      one CTA per (sample, head, 128-query tile), 8 warps x 16 query rows; K/V windows stream.
//   attn_delta_tiled_kernel    delta = rowsum(dO (.) (O + O_lo)) -> the caller's delta_ws [B,H,N] (fixed-order shuffles).
//   attn_bwd_dq_tiled_kernel   one CTA per (sample, head, 64-query tile), 4 warps; Q/dO fragments, lse and delta in
//                              registers; K/V windows stream.
//   attn_bwd_dkdv_tiled_kernel one CTA per (sample, head, 64-key tile), 4 warps; K/V fragments in registers; Q, dO,
//                              lse and delta windows stream.
// No atomics: every dqkv element is written by one thread, so dqkv is bit-identical from run to run.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "attention_mma.cuh"
#include "kernels.h"

namespace cara {
namespace {

constexpr int TD = 80;                     // head size
using Tile = HeadTile<TD>;
constexpr int TP = Tile::PITCH;            // 176-byte rows
constexpr int WIN = 64;                    // rows per streamed window = one chunk of the chunk functions
static_assert(WIN == KC && WIN == QC, "a window is one chunk");

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory"); }

// rows [r0, r0 + ROWS) of one of q/k/v (or dO) of a head -> ROWS tile rows at dst.  Rows >= N are zero-filled through
// the src-size operand, with the source address clamped to the head's row 0: nothing is read from the next sample.
template <int ROWS>
__device__ __forceinline__ void load_rows(uint32_t dst, const __nv_bfloat16* src, long row_pitch, int r0, int N,
                                          int tid, int nthreads) {
  constexpr int CH = TD / 8;
  for (int idx = tid; idx < ROWS * CH; idx += nthreads) {
    const int row = idx / CH, ch = idx % CH, r = r0 + row;
    const bool ok = r < N;
    cp_async16(dst + row * TP + ch * 16, src + static_cast<long>(ok ? r : 0) * row_pitch + ch * 8, ok);
  }
}

// a tile holding rows [first, first + n) of the head at shared address w, addressed by absolute row (D = 80 tiles have
// no row swizzle, so shifting the base is all it takes)
__device__ __forceinline__ Tile window(uint32_t w, int first) { return Tile{w - static_cast<uint32_t>(first * TP)}; }

// ------------------------------------------------------------------------------------ forward
constexpr int FWD_THREADS = 256, FWD_ROWS = 128;                       // 8 warps x 16 query rows
constexpr int FWD_STAGE = 2 * WIN * TP;                                 // K window, then V window
constexpr int FWD_SMEM = FWD_ROWS * TP + 2 * FWD_STAGE;                 // 67,584 B

__global__ void __launch_bounds__(FWD_THREADS, 2)                    // 128 registers, two CTAs per SM
attn_fwd_tiled_kernel(const AttnArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = a.N, npad = ((N + 15) / 16) * 16, nwin = (npad + WIN - 1) / WIN;
  const int ntiles = (N + FWD_ROWS - 1) / FWD_ROWS;
  const int bh = blockIdx.x / ntiles, q_first = (blockIdx.x % ntiles) * FWD_ROWS;
  const int b = bh / a.H, h = bh % a.H;
  const long pitch = 3L * a.H * TD;
  const __nv_bfloat16* base = a.qkv + static_cast<long>(b) * N * pitch + h * TD;
  const uint32_t sq = s_u32(smem), skv = sq + FWD_ROWS * TP;
  auto load_window = [&](int w) {
    const uint32_t st = skv + (w & 1) * FWD_STAGE;
    load_rows<WIN>(st, base + a.H * TD, pitch, w * WIN, N, tid, FWD_THREADS);
    load_rows<WIN>(st + WIN * TP, base + 2 * a.H * TD, pitch, w * WIN, N, tid, FWD_THREADS);
    cp_async_commit();
  };
  load_rows<FWD_ROWS>(sq, base, pitch, q_first, N, tid, FWD_THREADS);  // committed with window 0
  load_window(0);

  const float sl2 = a.scale * 1.4426950408889634f;
  const int qt = q_first / 16 + warp;
  const bool active = qt * 16 < N;                                      // warp-uniform
  uint32_t qf[TD / 16][4];
  float o[TD / 8][4];
#pragma unroll
  for (int j = 0; j < TD / 8; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
  float m_lo = -CUDART_INF_F, m_hi = -CUDART_INF_F, l_lo = 0.f, l_hi = 0.f;
  for (int w = 0; w < nwin; ++w) {
    if (w + 1 < nwin) {
      load_window(w + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (active) {
      if (w == 0) load_a_frags<TD>(window(sq, q_first), qt * 16, lane, qf);
      const int k0 = w * WIN;
      const uint32_t st = skv + (w & 1) * FWD_STAGE;
      const Tile tk = window(st, k0), tv = window(st + WIN * TP, k0);
      if (k0 + KC <= npad) {
        fwd_chunk<TD, KC / 16>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o);
      } else {
        switch ((npad - k0) / 16) {                                     // N is padded to 16 keys, not to the window
          case 1: fwd_chunk<TD, 1>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o); break;
          case 2: fwd_chunk<TD, 2>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o); break;
          case 3: fwd_chunk<TD, 3>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o); break;
          default: break;
        }
      }
    }
    __syncthreads();                                                    // the stage is refilled at w + 2
  }
  if (!active) return;

  // the epilogue of attn_fwd_kernel (attention.cu), unchanged
  const int g = lane >> 2, t = lane & 3;
  l_lo = quad_sum(l_lo); l_hi = quad_sum(l_hi);
  const float i_lo = 1.0f / l_lo, i_hi = 1.0f / l_hi;
  const int r_lo = qt * 16 + g, r_hi = r_lo + 8;
  const long obase = (static_cast<long>(b) * N) * (a.H * TD) + h * TD;
  auto put = [&](int row, int col, float v0, float v1) {
    const __nv_bfloat162 hi = __floats2bfloat162_rn(v0, v1);
    *reinterpret_cast<__nv_bfloat162*>(a.o + obase + static_cast<long>(row) * a.H * TD + col) = hi;
    if (a.o_lo != nullptr) {
      const float2 hf = __bfloat1622float2(hi);
      *reinterpret_cast<uint32_t*>(a.o_lo + obase + static_cast<long>(row) * a.H * TD + col) = pack2(v0 - hf.x, v1 - hf.y);
    }
  };
#pragma unroll
  for (int j = 0; j < TD / 8; ++j) {
    const int col = j * 8 + 2 * t;
    if (r_lo < N) put(r_lo, col, o[j][0] * i_lo, o[j][1] * i_lo);
    if (r_hi < N) put(r_hi, col, o[j][2] * i_hi, o[j][3] * i_hi);
  }
  if (a.lse != nullptr && t == 0) {
    float* lse = a.lse + (static_cast<long>(b) * a.H + h) * N;
    if (r_lo < N) lse[r_lo] = m_lo + log2f(l_lo);
    if (r_hi < N) lse[r_hi] = m_hi + log2f(l_hi);
  }
}

// ------------------------------------------------------------------------------------ backward
constexpr int DELTA_THREADS = 256;

// one CTA per (sample, head): the whole-head backward's delta loop, into global memory
__global__ void __launch_bounds__(DELTA_THREADS)
attn_delta_tiled_kernel(const AttnArgs a) {
  const int tid = threadIdx.x, lane = tid & 31;
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int N = a.N, C = a.H * TD;
  const long off = static_cast<long>(b) * N * C + h * TD;
  delta_rows<TD, DELTA_THREADS>(a.d_o + off, a.o + off, a.o_lo + off, C, N, tid, lane,
                                a.delta + (static_cast<long>(b) * a.H + h) * N);
}

constexpr int BWD_THREADS = 128, BWD_ROWS = 64;                         // 4 warps x 16 rows
constexpr int BWD_STAGE = 2 * WIN * TP;                                 // two operand windows
constexpr int DQ_SMEM = 2 * BWD_ROWS * TP + 2 * BWD_STAGE;              // Q, dO tiles + K/V ring: 67,584 B
constexpr int DKDV_SMEM = 2 * BWD_ROWS * TP + 2 * BWD_STAGE + 2 * 2 * WIN * 4;   // K, V tiles + Q/dO ring + lse/delta

__global__ void __launch_bounds__(BWD_THREADS)
attn_bwd_dq_tiled_kernel(const AttnArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = a.N, npad = ((N + 15) / 16) * 16, nwin = (npad + WIN - 1) / WIN;
  const int ntiles = (N + BWD_ROWS - 1) / BWD_ROWS;
  const int bh = blockIdx.x / ntiles, q_first = (blockIdx.x % ntiles) * BWD_ROWS;
  const int b = bh / a.H, h = bh % a.H;
  const int C = a.H * TD;
  const long pitch = 3L * C;
  const __nv_bfloat16* base = a.qkv + static_cast<long>(b) * N * pitch + h * TD;
  const __nv_bfloat16* dob = a.d_o + static_cast<long>(b) * N * C + h * TD;
  const uint32_t sq = s_u32(smem), sdo = sq + BWD_ROWS * TP, skv = sdo + BWD_ROWS * TP;
  auto load_window = [&](int w) {
    const uint32_t st = skv + (w & 1) * BWD_STAGE;
    load_rows<WIN>(st, base + C, pitch, w * WIN, N, tid, BWD_THREADS);
    load_rows<WIN>(st + WIN * TP, base + 2 * C, pitch, w * WIN, N, tid, BWD_THREADS);
    cp_async_commit();
  };
  load_rows<BWD_ROWS>(sq, base, pitch, q_first, N, tid, BWD_THREADS);  // committed with window 0
  load_rows<BWD_ROWS>(sdo, dob, C, q_first, N, tid, BWD_THREADS);
  load_window(0);

  const float sl2 = a.scale * 1.4426950408889634f;
  const int g = lane >> 2, t = lane & 3;
  const int qt = q_first / 16 + warp;
  const bool active = qt * 16 < N;
  const int r_lo = qt * 16 + g, r_hi = r_lo + 8;
  // rows >= N as in the whole-head kernel's shared statistics (their dq is not written)
  const long srow = (static_cast<long>(b) * a.H + h) * N;
  const float lse_lo = r_lo < N ? a.lse[srow + r_lo] : 1e30f, lse_hi = r_hi < N ? a.lse[srow + r_hi] : 1e30f;
  const float dl_lo = r_lo < N ? a.delta[srow + r_lo] : 0.f, dl_hi = r_hi < N ? a.delta[srow + r_hi] : 0.f;
  uint32_t qf[TD / 16][4], dof[TD / 16][4];
  float dq[TD / 8][4];
#pragma unroll
  for (int j = 0; j < TD / 8; ++j) dq[j][0] = dq[j][1] = dq[j][2] = dq[j][3] = 0.f;
  for (int w = 0; w < nwin; ++w) {
    if (w + 1 < nwin) {
      load_window(w + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (active) {
      if (w == 0) {
        load_a_frags<TD>(window(sq, q_first), qt * 16, lane, qf);
        load_a_frags<TD>(window(sdo, q_first), qt * 16, lane, dof);
      }
      const int k0 = w * WIN;
      const uint32_t st = skv + (w & 1) * BWD_STAGE;
      const Tile tk = window(st, k0), tv = window(st + WIN * TP, k0);
      if (k0 + KC <= npad) {
        dq_chunk<TD, KC / 16>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq);
      } else {
        switch ((npad - k0) / 16) {
          case 1: dq_chunk<TD, 1>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq); break;
          case 2: dq_chunk<TD, 2>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq); break;
          case 3: dq_chunk<TD, 3>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq); break;
          default: break;
        }
      }
    }
    __syncthreads();
  }
  if (!active) return;
  __nv_bfloat16* dq_base = a.dqkv + static_cast<long>(b) * N * pitch + h * TD;
#pragma unroll
  for (int j = 0; j < TD / 8; ++j) {
    const int col = j * 8 + 2 * t;
    if (r_lo < N) *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_lo) * pitch + col) = pack2(dq[j][0] * a.scale, dq[j][1] * a.scale);
    if (r_hi < N) *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_hi) * pitch + col) = pack2(dq[j][2] * a.scale, dq[j][3] * a.scale);
  }
}

__global__ void __launch_bounds__(BWD_THREADS)
attn_bwd_dkdv_tiled_kernel(const AttnArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = a.N, npad = ((N + 15) / 16) * 16, nwin = (npad + WIN - 1) / WIN;
  const int ntiles = (N + BWD_ROWS - 1) / BWD_ROWS;
  const int bh = blockIdx.x / ntiles, k_first = (blockIdx.x % ntiles) * BWD_ROWS;
  const int b = bh / a.H, h = bh % a.H;
  const int C = a.H * TD;
  const long pitch = 3L * C;
  const __nv_bfloat16* base = a.qkv + static_cast<long>(b) * N * pitch + h * TD;
  const __nv_bfloat16* dob = a.d_o + static_cast<long>(b) * N * C + h * TD;
  const long srow = (static_cast<long>(b) * a.H + h) * N;
  const uint32_t sk = s_u32(smem), sv = sk + BWD_ROWS * TP, sqd = sv + BWD_ROWS * TP;
  float* s_stat = reinterpret_cast<float*>(smem + 2 * BWD_ROWS * TP + 2 * BWD_STAGE);   // per stage: lse[WIN], delta[WIN]
  auto load_window = [&](int w) {
    const int s = w & 1, q0 = w * WIN;
    const uint32_t st = sqd + s * BWD_STAGE;
    load_rows<WIN>(st, base, pitch, q0, N, tid, BWD_THREADS);
    load_rows<WIN>(st + WIN * TP, dob, C, q0, N, tid, BWD_THREADS);
    cp_async_commit();
    // padded query rows get lse = +big (P = 0) and delta = 0, as in the whole-head kernel
    for (int i = tid; i < WIN; i += BWD_THREADS) {
      const int q = q0 + i;
      s_stat[s * 2 * WIN + i] = q < N ? a.lse[srow + q] : 1e30f;
      s_stat[s * 2 * WIN + WIN + i] = q < N ? a.delta[srow + q] : 0.f;
    }
  };
  load_rows<BWD_ROWS>(sk, base + C, pitch, k_first, N, tid, BWD_THREADS);   // committed with window 0
  load_rows<BWD_ROWS>(sv, base + 2 * C, pitch, k_first, N, tid, BWD_THREADS);
  load_window(0);

  const float sl2 = a.scale * 1.4426950408889634f;
  const int g = lane >> 2, t = lane & 3;
  const int kt = k_first / 16 + warp;
  const bool active = kt * 16 < N;
  uint32_t kf[TD / 16][4], vf[TD / 16][4];
  float dk[TD / 8][4], dv[TD / 8][4];
#pragma unroll
  for (int j = 0; j < TD / 8; ++j) {
    dk[j][0] = dk[j][1] = dk[j][2] = dk[j][3] = 0.f;
    dv[j][0] = dv[j][1] = dv[j][2] = dv[j][3] = 0.f;
  }
  for (int w = 0; w < nwin; ++w) {
    if (w + 1 < nwin) {
      load_window(w + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (active) {
      if (w == 0) {
        load_a_frags<TD>(window(sk, k_first), kt * 16, lane, kf);
        load_a_frags<TD>(window(sv, k_first), kt * 16, lane, vf);
      }
      const int q0 = w * WIN, s = w & 1;
      const uint32_t st = sqd + s * BWD_STAGE;
      const Tile tq = window(st, q0), tdo = window(st + WIN * TP, q0);
      const float* s_lse = s_stat + s * 2 * WIN - q0;                  // indexed by absolute query row
      const float* s_delta = s_lse + WIN;
      if (q0 + QC <= npad) {
        dkdv_chunk<TD, QC / 16>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv);
      } else {
        switch ((npad - q0) / 16) {
          case 1: dkdv_chunk<TD, 1>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv); break;
          case 2: dkdv_chunk<TD, 2>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv); break;
          case 3: dkdv_chunk<TD, 3>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv); break;
          default: break;
        }
      }
    }
    __syncthreads();
  }
  if (!active) return;
  __nv_bfloat16* dq_base = a.dqkv + static_cast<long>(b) * N * pitch + h * TD;
  const int r_lo = kt * 16 + g, r_hi = r_lo + 8;
#pragma unroll
  for (int j = 0; j < TD / 8; ++j) {
    const int col = j * 8 + 2 * t;
    if (r_lo < N) {
      *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_lo) * pitch + C + col) = pack2(dk[j][0] * a.scale, dk[j][1] * a.scale);
      *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_lo) * pitch + 2 * C + col) = pack2(dv[j][0], dv[j][1]);
    }
    if (r_hi < N) {
      *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_hi) * pitch + C + col) = pack2(dk[j][2] * a.scale, dk[j][3] * a.scale);
      *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_hi) * pitch + 2 * C + col) = pack2(dv[j][2], dv[j][3]);
    }
  }
}

template <typename Kern>
int raise_smem(Kern kernel, int smem, bool& configured) {
  if (!configured) {
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -52;
    configured = true;
  }
  return 0;
}

}  // namespace

int attn_fwd_tiled_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.D != TD || a.B <= 0 || a.N <= 0 || a.H <= 0 || a.qkv == nullptr || a.o == nullptr) return -50;
  static bool configured = false;
  if (const int rc = raise_smem(attn_fwd_tiled_kernel, FWD_SMEM, configured)) return rc;
  const long grid = static_cast<long>(a.B) * a.H * ((a.N + FWD_ROWS - 1) / FWD_ROWS);
  if (grid > 0x7fffffffL) return -50;
  attn_fwd_tiled_kernel<<<static_cast<unsigned>(grid), FWD_THREADS, FWD_SMEM, st>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : -53;
}

int attn_bwd_tiled_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.D != TD || a.B <= 0 || a.N <= 0 || a.H <= 0) return -50;
  if (a.qkv == nullptr || a.o == nullptr || a.o_lo == nullptr || a.lse == nullptr || a.d_o == nullptr ||
      a.dqkv == nullptr || a.delta == nullptr)
    return -50;
  static bool dq_configured = false, dkdv_configured = false;
  if (const int rc = raise_smem(attn_bwd_dq_tiled_kernel, DQ_SMEM, dq_configured)) return rc;
  if (const int rc = raise_smem(attn_bwd_dkdv_tiled_kernel, DKDV_SMEM, dkdv_configured)) return rc;
  const long grid = static_cast<long>(a.B) * a.H * ((a.N + BWD_ROWS - 1) / BWD_ROWS);
  if (grid > 0x7fffffffL) return -50;
  attn_delta_tiled_kernel<<<a.B * a.H, DELTA_THREADS, 0, st>>>(a);
  attn_bwd_dq_tiled_kernel<<<static_cast<unsigned>(grid), BWD_THREADS, DQ_SMEM, st>>>(a);
  attn_bwd_dkdv_tiled_kernel<<<static_cast<unsigned>(grid), BWD_THREADS, DKDV_SMEM, st>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : -53;
}

}  // namespace cara
