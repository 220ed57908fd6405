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
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdlib.h>

#include "kernels.h"

namespace cara {
namespace {

__device__ __forceinline__ uint32_t s_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool pred) {
  const int n = pred ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// Shared-memory tile of one head, conflict-free for ldmatrix (eight 16-byte rows per phase must fall in distinct
// bank groups): D = 64 -> dense 128-byte rows with the 16-byte chunk index XOR-swizzled by (row & 7), so four
// tiles of 208 rows fit twice per SM; other D -> rows padded by 16 B (pitch mod 128 = 48 for D = 80).
template <int D>
struct HeadTile {
  static constexpr int PITCH = D == 64 ? 128 : D * 2 + 16;
  uint32_t base;
  __device__ __forceinline__ uint32_t at(int row, int chunk16) const {
    if (D == 64) return base + row * 128 + ((chunk16 ^ (row & 7)) << 4);
    return base + row * PITCH + chunk16 * 16;
  }
};

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

// A-operand fragments (16 rows x D) of a row-major tile: DK k-steps of 4 registers
template <int D>
__device__ __forceinline__ void load_a_frags(const HeadTile<D>& t, int row0, int lane, uint32_t (&f)[D / 16][4]) {
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk) ldsm_x4(t.at(row0 + (lane & 15), kk * 2 + (lane >> 4)), f[kk]);
}

// acc[j] (16 x 8 tiles, j over NT column tiles starting at row col0 of `t`) += A(16 x D) * t[col rows]^T
template <int D, int NT>
__device__ __forceinline__ void mma_a_bt(const uint32_t (&af)[D / 16][4], const HeadTile<D>& t, int col0, int lane,
                                         float (&acc)[NT][4]) {
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk) {
#pragma unroll
    for (int jp = 0; jp < NT / 2; ++jp) {
      uint32_t bf[4];
      const int n = col0 + jp * 16 + (lane & 7) + ((lane >> 4) & 1) * 8;
      ldsm_x4(t.at(n, kk * 2 + ((lane >> 3) & 1)), bf);
      mma_bf16(acc[jp * 2 + 0], af[kk], bf[0], bf[1]);
      mma_bf16(acc[jp * 2 + 1], af[kk], bf[2], bf[3]);
    }
  }
}

// out[j] (16 x 8 tiles over D) += P(16 x 8*NT, fp32 accumulator layout, converted to bf16) * t[rows k0..]
template <int D, int NT>
__device__ __forceinline__ void mma_p_b(const float (&p)[NT][4], const HeadTile<D>& t, int k0, int lane,
                                        float (&out)[D / 8][4]) {
  const int q = lane >> 3;
#pragma unroll
  for (int ks = 0; ks < NT / 2; ++ks) {
    uint32_t af[4];
    af[0] = pack2(p[2 * ks][0], p[2 * ks][1]);
    af[1] = pack2(p[2 * ks][2], p[2 * ks][3]);
    af[2] = pack2(p[2 * ks + 1][0], p[2 * ks + 1][1]);
    af[3] = pack2(p[2 * ks + 1][2], p[2 * ks + 1][3]);
#pragma unroll
    for (int jp = 0; jp < D / 16; ++jp) {
      uint32_t bf[4];
      ldsm_x4_t(t.at(k0 + ks * 16 + (lane & 7) + (q & 1) * 8, jp * 2 + (q >> 1)), bf);
      mma_bf16(out[jp * 2 + 0], af, bf[0], bf[1]);
      mma_bf16(out[jp * 2 + 1], af, bf[2], bf[3]);
    }
  }
}

constexpr int KC = 64;   // keys per chunk (forward and dQ pass)
constexpr int QC = 64;   // queries per chunk (dK/dV pass)

// one chunk of NTP*16 keys of the forward: S = Q K^T, online softmax update, O += P V
template <int D, int NTP>
__device__ __forceinline__ void fwd_chunk(const uint32_t (&qf)[D / 16][4], const HeadTile<D>& tk, const HeadTile<D>& tv,
                                          int k0, int N, int lane, float sl2, float& m_lo, float& m_hi, float& l_lo,
                                          float& l_hi, float (&o)[D / 8][4]) {
  constexpr int NT = NTP * 2;
  const int t = lane & 3;
  float s[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
  mma_a_bt<D, NT>(qf, tk, k0, lane, s);
  float mx_lo = m_lo, mx_hi = m_hi;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int key = k0 + j * 8 + 2 * t;
    s[j][0] = key < N ? s[j][0] * sl2 : -CUDART_INF_F;
    s[j][1] = key + 1 < N ? s[j][1] * sl2 : -CUDART_INF_F;
    s[j][2] = key < N ? s[j][2] * sl2 : -CUDART_INF_F;
    s[j][3] = key + 1 < N ? s[j][3] * sl2 : -CUDART_INF_F;
    mx_lo = fmaxf(mx_lo, fmaxf(s[j][0], s[j][1]));
    mx_hi = fmaxf(mx_hi, fmaxf(s[j][2], s[j][3]));
  }
  mx_lo = quad_max(mx_lo); mx_hi = quad_max(mx_hi);      // finite: chunk 0 always holds key 0
  const float c_lo = exp2f(m_lo - mx_lo), c_hi = exp2f(m_hi - mx_hi);
  m_lo = mx_lo; m_hi = mx_hi;
  l_lo *= c_lo; l_hi *= c_hi;
#pragma unroll
  for (int j = 0; j < D / 8; ++j) { o[j][0] *= c_lo; o[j][1] *= c_lo; o[j][2] *= c_hi; o[j][3] *= c_hi; }
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    s[j][0] = exp2f(s[j][0] - m_lo); s[j][1] = exp2f(s[j][1] - m_lo);
    s[j][2] = exp2f(s[j][2] - m_hi); s[j][3] = exp2f(s[j][3] - m_hi);
    l_lo += s[j][0] + s[j][1]; l_hi += s[j][2] + s[j][3];
  }
  mma_p_b<D, NT>(s, tv, k0, lane, o);
}

// one chunk of NTP*16 keys of the dQ pass: recompute P, dP; dS = P (.) (dP - delta); dQ += dS K
template <int D, int NTP>
__device__ __forceinline__ void dq_chunk(const uint32_t (&qf)[D / 16][4], const uint32_t (&dof)[D / 16][4],
                                         const HeadTile<D>& tk, const HeadTile<D>& tv, int k0, int N, int lane,
                                         float sl2, float lse_lo, float lse_hi, float dl_lo, float dl_hi,
                                         float (&dq)[D / 8][4]) {
  constexpr int NT = NTP * 2;
  const int t = lane & 3;
  float s[NT][4], dp[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
    dp[j][0] = dp[j][1] = dp[j][2] = dp[j][3] = 0.f;
  }
  mma_a_bt<D, NT>(qf, tk, k0, lane, s);
  mma_a_bt<D, NT>(dof, tv, k0, lane, dp);
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int key = k0 + j * 8 + 2 * t;
    const float p0 = key < N ? exp2f(s[j][0] * sl2 - lse_lo) : 0.f;
    const float p1 = key + 1 < N ? exp2f(s[j][1] * sl2 - lse_lo) : 0.f;
    const float p2 = key < N ? exp2f(s[j][2] * sl2 - lse_hi) : 0.f;
    const float p3 = key + 1 < N ? exp2f(s[j][3] * sl2 - lse_hi) : 0.f;
    s[j][0] = p0 * (dp[j][0] - dl_lo); s[j][1] = p1 * (dp[j][1] - dl_lo);
    s[j][2] = p2 * (dp[j][2] - dl_hi); s[j][3] = p3 * (dp[j][3] - dl_hi);
  }
  mma_p_b<D, NT>(s, tk, k0, lane, dq);
}

// one chunk of NTP*16 queries of the dK/dV pass (transposed tiles: rows = keys, columns = queries)
template <int D, int NTP>
__device__ __forceinline__ void dkdv_chunk(const uint32_t (&kf)[D / 16][4], const uint32_t (&vf)[D / 16][4],
                                           const HeadTile<D>& tq, const HeadTile<D>& tdo, int q0, int lane, float sl2,
                                           const float* s_lse, const float* s_delta, float (&dk)[D / 8][4],
                                           float (&dv)[D / 8][4]) {
  constexpr int NT = NTP * 2;
  const int t = lane & 3;
  float st[NT][4], dpt[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    st[j][0] = st[j][1] = st[j][2] = st[j][3] = 0.f;
    dpt[j][0] = dpt[j][1] = dpt[j][2] = dpt[j][3] = 0.f;
  }
  mma_a_bt<D, NT>(kf, tq, q0, lane, st);      // S^T = K Q^T
  mma_a_bt<D, NT>(vf, tdo, q0, lane, dpt);    // dP^T = V dO^T
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int qi = q0 + j * 8 + 2 * t;
    const float l0 = s_lse[qi], l1 = s_lse[qi + 1], d0 = s_delta[qi], d1 = s_delta[qi + 1];
    const float p0 = exp2f(st[j][0] * sl2 - l0), p1 = exp2f(st[j][1] * sl2 - l1);
    const float p2 = exp2f(st[j][2] * sl2 - l0), p3 = exp2f(st[j][3] * sl2 - l1);
    dpt[j][0] = p0 * (dpt[j][0] - d0); dpt[j][1] = p1 * (dpt[j][1] - d1);
    dpt[j][2] = p2 * (dpt[j][2] - d0); dpt[j][3] = p3 * (dpt[j][3] - d1);
    st[j][0] = p0; st[j][1] = p1; st[j][2] = p2; st[j][3] = p3;
  }
  mma_p_b<D, NT>(st, tdo, q0, lane, dv);      // dV += P^T dO
  mma_p_b<D, NT>(dpt, tq, q0, lane, dk);      // dK += dS^T Q
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
  {
    // One group of G lanes per row: lane c of the group loads 16-byte chunk c of the row, and the group sums the
    // chunks with shuffles in a fixed order, so dqkv is bit-identical from run to run (shared-memory atomics from
    // several warps into one row -- a D = 80 row spans two warps -- add in whatever order the warps arrive).
    // U rows in flight per group, 32 per pass of the CTA: this loop is the global-latency part of the CTA.
    constexpr int CH = D / 8, G = CH <= 8 ? 8 : 16, U = G / 4, NG = BWD_THREADS / G;
    static_assert(CH <= 16, "one row per group of at most 16 lanes");
    const int c = lane % G, grp = tid / G;
    auto dot8 = [](const uint4& x, const uint4& y, const uint4& z) {
      const uint32_t xw[4] = {x.x, x.y, x.z, x.w}, yw[4] = {y.x, y.y, y.z, y.w}, zw[4] = {z.x, z.y, z.z, z.w};
      float acc = 0.f;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 xf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&xw[e]));
        const float2 yf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&yw[e]));
        const float2 zf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&zw[e]));
        acc += xf.x * (yf.x + zf.x) + xf.y * (yf.y + zf.y);
      }
      return acc;
    };
    for (int r0 = 0; r0 < N; r0 += U * NG) {                   // warp-uniform trip count: every lane shuffles
      uint4 x[U] = {}, y[U] = {}, z[U] = {};
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int r = r0 + u * NG + grp;
        if (c < CH && r < N) {
          const long off = static_cast<long>(r) * C + c * 8;
          x[u] = *reinterpret_cast<const uint4*>(dob + off);
          y[u] = *reinterpret_cast<const uint4*>(ob + off);
          z[u] = *reinterpret_cast<const uint4*>(olb + off);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float v = dot8(x[u], y[u], z[u]);                         // 0 for idle lanes and rows >= N
#pragma unroll
        for (int s = G / 2; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
        const int r = r0 + u * NG + grp;
        if (c == 0 && r < N) s_delta[r] = v;
      }
    }
  }
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
