// Attention core of cp_attn (cara.py:44-48): softmax(q k^T * D^-1/2) v and its backward, one CTA per
// (sample, head).  N is 197 (ViT-B/L @224/16) or 257 (ViT-H/14): the whole head's K/V (and Q/dO in the
// backward) live in shared memory, the [N,N] score matrix never touches HBM (the reference round-trips
// 3072 x 197 x 197 fp32 = 477 MB per layer at batch 256, SURVEY row a2).
//
// q/k/v are read in place from the fused projection's [B, N, 3, H, D] output and o is written as
// [B, N, H, D] -- the permute/transpose copies of cara.py:36-41,48 disappear.
//
// Math: warp-level mma.sync m16n8k16 bf16 with fp32 accumulation, flash-style online softmax over
// 64-key chunks (exp2 with pre-scaled logits), fp32 softmax statistics.  Backward is two passes over
// the head held in shared memory (warps own query tiles for delta + dQ, then key tiles for dK/dV) so no
// atomics are needed; delta = rowsum(dO (.) O) uses O kept as a bf16 (hi, lo) pair.  Attention is ~6 % of the step's FLOPs (SURVEY Appendix C).
// The chunk functions live in attention_mma.cuh; the key-tiled D = 80 kernels of attention_tiled.cu run them for N
// beyond the shared-memory limits of these kernels (forward N <= 432, backward N <= 320 at D = 80).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdlib.h>

#include "attention_mma.cuh"
#include "kernels.h"

namespace cara {
namespace {

__device__ __forceinline__ void cp_async_commit_wait_all() {
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// cooperative load of rows [0, npad) of one of q/k/v (or dO) for head (b,h); rows >= N are zero-filled
template <int D>
__device__ __forceinline__ void load_head(const HeadTile<D>& t, const __nv_bfloat16* src, long row_pitch, int N,
                                          int npad, int tid, int nthreads) {
  constexpr int CH = D / 8;
  for (int idx = tid; idx < npad * CH; idx += nthreads) {
    const int row = idx / CH, ch = idx % CH;
    const bool ok = row < N;
    cp_async16(t.at(row, ch), src + static_cast<long>(ok ? row : 0) * row_pitch + ch * 8, ok);
  }
}

// ------------------------------------------------------------------------------------ forward
constexpr int FWD_THREADS = 256;

template <int D>
__global__ void __launch_bounds__(FWD_THREADS, D == 64 ? 2 : 1)
attn_fwd_kernel(const AttnArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int N = a.N, npad = ((N + 15) / 16) * 16;
  const long pitch = 3L * a.H * D;
  const __nv_bfloat16* base = a.qkv + static_cast<long>(b) * N * pitch + h * D;
  HeadTile<D> tq{s_u32(smem)}, tk{tq.base + npad * HeadTile<D>::PITCH}, tv{tk.base + npad * HeadTile<D>::PITCH};
  load_head<D>(tq, base, pitch, N, npad, tid, FWD_THREADS);
  load_head<D>(tk, base + a.H * D, pitch, N, npad, tid, FWD_THREADS);
  load_head<D>(tv, base + 2 * a.H * D, pitch, N, npad, tid, FWD_THREADS);
  cp_async_commit_wait_all();
  __syncthreads();

  const float sl2 = a.scale * 1.4426950408889634f;
  const int g = lane >> 2, t = lane & 3;
  for (int qt = warp; qt * 16 < N; qt += FWD_THREADS / 32) {
    uint32_t qf[D / 16][4];
    load_a_frags<D>(tq, qt * 16, lane, qf);
    float o[D / 8][4];
#pragma unroll
    for (int j = 0; j < D / 8; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
    float m_lo = -CUDART_INF_F, m_hi = -CUDART_INF_F, l_lo = 0.f, l_hi = 0.f;
    int k0 = 0;
    for (; k0 + KC <= npad; k0 += KC) fwd_chunk<D, KC / 16>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o);
    switch ((npad - k0) / 16) {                    // N is padded to 16 keys, not to the chunk size
      case 1: fwd_chunk<D, 1>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o); break;
      case 2: fwd_chunk<D, 2>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o); break;
      case 3: fwd_chunk<D, 3>(qf, tk, tv, k0, N, lane, sl2, m_lo, m_hi, l_lo, l_hi, o); break;
      default: break;
    }
    l_lo = quad_sum(l_lo); l_hi = quad_sum(l_hi);
    const float i_lo = 1.0f / l_lo, i_hi = 1.0f / l_hi;
    const int r_lo = qt * 16 + g, r_hi = r_lo + 8;
    const long obase = (static_cast<long>(b) * N) * (a.H * D) + h * D;
    // o (bf16) feeds the output projection; o_lo = bf16(o_fp32 - o) is kept for backward so that
    // delta = rowsum(dO (.) O) is formed from a ~16-bit-mantissa O (see attn_bwd_kernel)
    auto put = [&](int row, int col, float v0, float v1) {
      const __nv_bfloat162 hi = __floats2bfloat162_rn(v0, v1);
      *reinterpret_cast<__nv_bfloat162*>(a.o + obase + static_cast<long>(row) * a.H * D + col) = hi;
      if (a.o_lo != nullptr) {
        const float2 hf = __bfloat1622float2(hi);
        *reinterpret_cast<uint32_t*>(a.o_lo + obase + static_cast<long>(row) * a.H * D + col) = pack2(v0 - hf.x, v1 - hf.y);
      }
    };
#pragma unroll
    for (int j = 0; j < D / 8; ++j) {
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
}

// ------------------------------------------------------------------------------------ backward
constexpr int BWD_THREADS = 128;

template <int D>
__global__ void __launch_bounds__(BWD_THREADS, D == 64 ? 2 : 1)
attn_bwd_kernel(const AttnArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int NW = BWD_THREADS / 32;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int N = a.N, npad = ((N + 15) / 16) * 16, nstat = ((N + QC - 1) / QC) * QC;
  const int C = a.H * D;
  const long pitch = 3L * C;
  const __nv_bfloat16* base = a.qkv + static_cast<long>(b) * N * pitch + h * D;
  const __nv_bfloat16* dob = a.d_o + static_cast<long>(b) * N * C + h * D;
  const __nv_bfloat16* ob = a.o + static_cast<long>(b) * N * C + h * D;
  const __nv_bfloat16* olb = a.o_lo + static_cast<long>(b) * N * C + h * D;
  constexpr int TB = HeadTile<D>::PITCH;
  HeadTile<D> tq{s_u32(smem)}, tk{tq.base + npad * TB}, tv{tk.base + npad * TB}, tdo{tv.base + npad * TB};
  float* s_lse = reinterpret_cast<float*>(smem + 4 * npad * TB);
  float* s_delta = s_lse + nstat;
  load_head<D>(tq, base, pitch, N, npad, tid, BWD_THREADS);
  load_head<D>(tk, base + C, pitch, N, npad, tid, BWD_THREADS);
  load_head<D>(tv, base + 2 * C, pitch, N, npad, tid, BWD_THREADS);
  load_head<D>(tdo, dob, C, N, npad, tid, BWD_THREADS);
  // delta_i = sum_d dO[i,d] (O + O_lo)[i,d]: O carried as a bf16 (hi, lo) pair, because with the plain bf16 O
  // the rounding of O is the dominant dq/dk error for peaked softmax rows (rows of dS no longer sum to ~0).
  // lse padded with +big so padded queries get P = 0 in pass 2.
  const float* lse = a.lse + (static_cast<long>(b) * a.H + h) * N;
  for (int row = tid; row < nstat; row += BWD_THREADS) {
    s_lse[row] = row < N ? lse[row] : 1e30f;
    if (row >= N) s_delta[row] = 0.f;
  }
  delta_rows<D, BWD_THREADS>(dob, ob, olb, C, N, tid, lane, s_delta);
  cp_async_commit_wait_all();
  __syncthreads();

  const float sl2 = a.scale * 1.4426950408889634f;
  const int g = lane >> 2, t = lane & 3;
  __nv_bfloat16* dq_base = a.dqkv + static_cast<long>(b) * N * pitch + h * D;

  // ---- pass 1: warps own 16-query tiles -> dQ
  for (int qt = warp; qt * 16 < N; qt += NW) {
    uint32_t qf[D / 16][4], dof[D / 16][4];
    load_a_frags<D>(tq, qt * 16, lane, qf);
    load_a_frags<D>(tdo, qt * 16, lane, dof);
    const int r_lo = qt * 16 + g, r_hi = r_lo + 8;
    const float lse_lo = s_lse[r_lo], lse_hi = s_lse[r_hi];
    const float dl_lo = s_delta[r_lo], dl_hi = s_delta[r_hi];
    float dq[D / 8][4];
#pragma unroll
    for (int j = 0; j < D / 8; ++j) dq[j][0] = dq[j][1] = dq[j][2] = dq[j][3] = 0.f;
    int k0 = 0;
    for (; k0 + KC <= npad; k0 += KC)
      dq_chunk<D, KC / 16>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq);
    switch ((npad - k0) / 16) {
      case 1: dq_chunk<D, 1>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq); break;
      case 2: dq_chunk<D, 2>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq); break;
      case 3: dq_chunk<D, 3>(qf, dof, tk, tv, k0, N, lane, sl2, lse_lo, lse_hi, dl_lo, dl_hi, dq); break;
      default: break;
    }
#pragma unroll
    for (int j = 0; j < D / 8; ++j) {
      const int col = j * 8 + 2 * t;
      if (r_lo < N) *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_lo) * pitch + col) = pack2(dq[j][0] * a.scale, dq[j][1] * a.scale);
      if (r_hi < N) *reinterpret_cast<uint32_t*>(dq_base + static_cast<long>(r_hi) * pitch + col) = pack2(dq[j][2] * a.scale, dq[j][3] * a.scale);
    }
  }

  // ---- pass 2: warps own 16-key tiles -> dK, dV (transposed score tiles: rows = keys, cols = queries)
  for (int kt = warp; kt * 16 < N; kt += NW) {
    uint32_t kf[D / 16][4], vf[D / 16][4];
    load_a_frags<D>(tk, kt * 16, lane, kf);
    load_a_frags<D>(tv, kt * 16, lane, vf);
    float dk[D / 8][4], dv[D / 8][4];
#pragma unroll
    for (int j = 0; j < D / 8; ++j) {
      dk[j][0] = dk[j][1] = dk[j][2] = dk[j][3] = 0.f;
      dv[j][0] = dv[j][1] = dv[j][2] = dv[j][3] = 0.f;
    }
    int q0 = 0;
    for (; q0 + QC <= npad; q0 += QC) dkdv_chunk<D, QC / 16>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv);
    switch ((npad - q0) / 16) {
      case 1: dkdv_chunk<D, 1>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv); break;
      case 2: dkdv_chunk<D, 2>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv); break;
      case 3: dkdv_chunk<D, 3>(kf, vf, tq, tdo, q0, lane, sl2, s_lse, s_delta, dk, dv); break;
      default: break;
    }
    const int r_lo = kt * 16 + g, r_hi = r_lo + 8;
#pragma unroll
    for (int j = 0; j < D / 8; ++j) {
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
}

template <int D>
int fwd_t(const AttnArgs& a, cudaStream_t st) {
  const int npad = ((a.N + 15) / 16) * 16;
  const int smem = 3 * npad * HeadTile<D>::PITCH;
  if (smem > 227 * 1024) return -51;
  static int configured = 0;
  if (configured < smem) {
    if (cudaFuncSetAttribute(attn_fwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -52;
    configured = smem;
  }
  attn_fwd_kernel<D><<<a.B * a.H, FWD_THREADS, smem, st>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : -53;
}
template <int D>
int bwd_t(const AttnArgs& a, cudaStream_t st) {
  const int npad = ((a.N + 15) / 16) * 16, nstat = ((a.N + QC - 1) / QC) * QC;
  const int smem = 4 * npad * HeadTile<D>::PITCH + 2 * nstat * 4;
  if (smem > 227 * 1024) return -51;
  static int configured = 0;
  if (configured < smem) {
    if (cudaFuncSetAttribute(attn_bwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -52;
    configured = smem;
  }
  attn_bwd_kernel<D><<<a.B * a.H, BWD_THREADS, smem, st>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : -53;
}

}  // namespace

// CARA_ATTN_TC (default 3): bit 0 = tcgen05 forward, bit 1 = tcgen05 backward (D = 64: attention_tc.cu for N <= 256,
// the key-tiled kernels of attention_long.cu above); D = 80 and cleared bits run the mma.sync kernels above.
static int attn_tc_mask() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("CARA_ATTN_TC");
    v = e != nullptr ? atoi(e) : 3;
  }
  return v;
}

int attn_fwd_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.B <= 0 || a.N <= 0 || a.H <= 0) return -50;
  if (attn_tc_mask() & 1) {
    int rc = attn_fwd_tc_launch(a, st);
    if (rc == 1) rc = attn_fwd_long_launch(a, st);
    if (rc <= 0) return rc;
  }
  if (a.D == 64) return fwd_t<64>(a, st);
  if (a.D == 80) return fwd_t<80>(a, st);
  return -50;
}
int attn_bwd_launch(const AttnArgs& a, cudaStream_t st) {
  if (a.B <= 0 || a.N <= 0 || a.H <= 0) return -50;
  if (a.o == nullptr) {                                         // delta already in a.delta (EPI_DELTA of the proj dX GEMM)
    int rc = (attn_tc_mask() & 2) ? attn_bwd_tc_launch(a, st) : 1;
    if (rc == 1 && (attn_tc_mask() & 2)) rc = attn_bwd_long_launch(a, st);
    return rc == 1 ? -50 : rc;
  }
  if (a.o_lo == nullptr) return -50;
  if (attn_tc_mask() & 2) {
    int rc = attn_bwd_tc_launch(a, st);
    if (rc == 1) rc = attn_bwd_long_launch(a, st);
    if (rc <= 0) return rc;
  }
  if (a.D == 64) return bwd_t<64>(a, st);
  if (a.D == 80) return bwd_t<80>(a, st);
  return -50;
}

}  // namespace cara
