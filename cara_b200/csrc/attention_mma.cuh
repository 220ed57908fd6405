// mma.sync building blocks of the attention core, shared by the whole-head kernels (attention.cu) and the key-tiled
// D = 80 kernels (attention_tiled.cu).  The chunk functions work on one 64-key (forward, dQ) or 64-query (dK/dV) chunk at
// ABSOLUTE row indices of the head: they only see the rows of the chunk through a HeadTile, so a caller that holds a
// window of the head instead of the whole head passes a tile whose base is shifted back by the window's first row.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

namespace cara {
namespace {

__device__ __forceinline__ uint32_t s_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool pred) {
  const int n = pred ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
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

// delta_i = sum_d dO[i,d] (O + O_lo)[i,d] for the rows [0, N) of one head (dob / ob / olb point at its row 0, row pitch
// C) -> out[i].  One group of G lanes per row: lane c of the group loads 16-byte chunk c of the row, and the group sums
// the chunks with shuffles in a fixed order, so dqkv is bit-identical from run to run (shared-memory atomics from
// several warps into one row -- a D = 80 row spans two warps -- add in whatever order the warps arrive).
// U rows in flight per group, NTHREADS / G * U per pass of the CTA: this loop is the global-latency part of the CTA.
template <int D, int NTHREADS>
__device__ __forceinline__ void delta_rows(const __nv_bfloat16* dob, const __nv_bfloat16* ob, const __nv_bfloat16* olb,
                                           int C, int N, int tid, int lane, float* out) {
  constexpr int CH = D / 8, G = CH <= 8 ? 8 : 16, U = G / 4, NG = NTHREADS / G;
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
      if (c == 0 && r < N) out[r] = v;
    }
  }
}

}  // namespace
}  // namespace cara
