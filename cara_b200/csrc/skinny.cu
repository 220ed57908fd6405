// Tall-skinny contractions of the CP adapter (SURVEY Appendix A.1/A.2).  HBM-bound: each streams one
// [M, K] activation / gradient matrix exactly once through a cp.async ring and contracts it against a
// rank-R operand with warp-level mma.sync (the tensor pipe is irrelevant here -- bytes are the cost).
//
// Precision: the rank-R path has only R terms per output, so bf16 rounding of its operands does not average
// out the way it does over K = 768..5120 in the frozen GEMM.  Factors and low-rank activations are therefore
// carried as bf16 (hi, lo) pairs (x = hi + lo, ~16 mantissa bits): factor matrices arrive as [hi rows; lo rows],
// the two partial products are folded in fp32, and Uhat / dThat are emitted as [hi | lo | hi] column blocks so
// that the tcgen05 GEMM's adapter segment computes hi*Bhi + lo*Bhi + hi*Blo against [Bhi | Bhi | Blo].
//
// (The row-wise contractions can also run as side tiles INSIDE the tcgen05 projection GEMM -- gemm_sm100.cu, opt-in:
// measured level with these stand-alone passes in the step, profiles/r02_side_tiles.md; the K = C ones also run inside the
// LayerNorm kernels, ln_rows.cu, default on.)
//
//   rows_kernel (row-wise, K reduced):
//     fwd : T = X A                     [M,Rp] fp32 (saved),  Uhat_s = cs_s (.) T   [M,S*3Rp] bf16 (hi|lo|hi)
//     bwd : dU_s = G_s B  per slice s,  dThat = sum_s cs_s (.) dU_s  [M,3Rp] bf16 (hi|lo|hi),
//           dcs_s = sum_m dU_s (.) T    [S,Rp] fp32 (atomically accumulated)
//   cols_kernel (column-wise, M reduced):
//     out[k,:] += sum_m X[m,k] (Vhi + Vlo)[m, slice(k)]   (dA = X^T dThat,  dB = sum_s G_s^T Uhat_s)
//     colsum[k] += sum_m X[m,k]                          (adapter-bias gradient)
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "kernels.h"

namespace cara {

__device__ __forceinline__ uint32_t s_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool pred) {
  const int n = pred ? 16 : 0;  // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
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

// ------------------------------------------------------------------------------------ rows_kernel
// Every CTA owns the same number of rows (<= 128: eight warps x one 16-row MMA tile) and the grid is exactly
// CTAs-per-SM x SMs, so all SMs stream the same number of bytes: with 128-row tiles M = 50,432 gave 394 CTAs on 444
// slots, a third CTA on 98 SMs and the other 50 SMs idle for a third of the launch.
constexpr int R_BM = 128, R_BK = 64, R_STAGES = 3;   // 3 x 20 KB: three CTAs per SM
// Rp = 64 (RT = 8): two warps share each 16-row tile, one per 32-column half of the rank, so a warp holds as many
// accumulators as at Rp = 32 and a CTA covers 64 rows.  4 stages x 24 KB, <= 128 registers: two CTAs per SM.
template <int RT> struct RowsCfg {
  static constexpr int WH = RT > 4 ? 2 : 1;        // warps per 16-row tile
  static constexpr int RW = RT / WH;               // 8-column rank tiles per warp
  static constexpr int BM = R_BM / WH;             // rows per CTA
  static constexpr int STAGES = RT > 4 ? 4 : R_STAGES;
  static constexpr int CTAS = RT > 4 ? 2 : 3;      // resident CTAs per SM (registers and shared memory)
  static constexpr int SMEM = STAGES * (BM * R_BK * 2 + 2 * RT * 8 * R_BK * 2);
};

template <int RT, int CS>
__global__ void __launch_bounds__(256, RowsCfg<RT>::CTAS)
rows_kernel(const RowsArgs a) {
  using Cfg = RowsCfg<RT>;
  constexpr int RP = RT * 8;
  constexpr int WH = Cfg::WH, RW = Cfg::RW, BM = Cfg::BM, STAGES = Cfg::STAGES;
  constexpr int NT = 2 * RW;                       // n-tiles of this warp incl. the lo halves of the factor
  constexpr int XS_BYTES = BM * R_BK * 2;          // 16 KB (8 KB at Rp = 64)
  constexpr int FS_BYTES = 2 * RP * R_BK * 2;
  constexpr int ST_BYTES = XS_BYTES + FS_BYTES;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ float red[CS * RP];
  pdl_wait();
  pdl_trigger();
  const uint32_t sbase = s_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wrow = WH == 1 ? warp : (warp & 3);    // this warp's 16-row tile
  const int cb = WH == 1 ? 0 : (warp >> 2) * RW * 8;   // and its first rank column
  const int m0 = blockIdx.x * a.rows_per_cta;
  const int m_end = min(a.M, m0 + a.rows_per_cta);
  const int cps = a.kslice / R_BK;                 // chunks per slice
  const int nch = CS * cps;

  auto issue = [&](int i) {
    if (i < nch) {
      const uint32_t xs = sbase + (i % STAGES) * ST_BYTES, fs = xs + XS_BYTES;
      const int kcol = i * R_BK;                   // column in X
      const int fcol = (i % cps) * R_BK;           // column in Ft
#pragma unroll
      for (int j = 0; j < BM / 32; ++j) {
        const int idx = j * 256 + tid, row = idx >> 3, ch = idx & 7;
        const bool ok = (m0 + row) < m_end;
        const __nv_bfloat16* src = a.X + static_cast<size_t>(ok ? m0 + row : 0) * a.ldx + kcol + ch * 8;
        cp_async16(xs + row * 128 + ((ch ^ (row & 7)) << 4), src, ok);
      }
      for (int idx = tid; idx < 2 * RP * 8; idx += 256) {
        const int row = idx >> 3, ch = idx & 7;
        cp_async16(fs + row * 128 + ((ch ^ (row & 7)) << 4), a.Ft + static_cast<size_t>(row) * a.ldf + fcol + ch * 8, true);
      }
    }
    cp_async_commit();
  };

  const int g = lane >> 2, t = lane & 3;
  const int r_lo = m0 + wrow * 16 + g, r_hi = r_lo + 8;
  const bool ok_lo = r_lo < m_end, ok_hi = r_hi < m_end;
  // emit v as the bf16 column blocks [hi | lo | hi] at row pointer p (block pitch RP)
  auto emit = [&](__nv_bfloat16* p, int col, float v0, float v1) {
    const __nv_bfloat162 hi = __floats2bfloat162_rn(v0, v1);
    const float2 hf = __bfloat1622float2(hi);
    const uint32_t h = *reinterpret_cast<const uint32_t*>(&hi);
    *reinterpret_cast<uint32_t*>(p + col) = h;
    *reinterpret_cast<uint32_t*>(p + RP + col) = pack2(v0 - hf.x, v1 - hf.y);
    *reinterpret_cast<uint32_t*>(p + 2 * RP + col) = h;
  };

  // backward: the saved T rows of this thread and the running dThat = sum_s cs_s (.) dU_s
  float2 t_lo[RW], t_hi[RW];
  float d[RW][4];
  if (a.mode != 0) {
    for (int i = tid; i < CS * RP; i += 256) red[i] = 0.f;
#pragma unroll
    for (int j = 0; j < RW; ++j) {
      const int col = cb + j * 8 + 2 * t;
      t_lo[j] = ok_lo ? *reinterpret_cast<const float2*>(a.T + static_cast<size_t>(r_lo) * RP + col) : make_float2(0.f, 0.f);
      t_hi[j] = ok_hi ? *reinterpret_cast<const float2*>(a.T + static_cast<size_t>(r_hi) * RP + col) : make_float2(0.f, 0.f);
      d[j][0] = d[j][1] = d[j][2] = d[j][3] = 0.f;
    }
  }

  for (int i = 0; i < STAGES - 1; ++i) issue(i);

  // one slice at a time through ONE set of accumulators (CS x fewer registers: three CTAs per SM for every CS)
#pragma unroll 1
  for (int s = 0; s < CS; ++s) {
    float acc[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] = 0.f;
    for (int c = 0; c < cps; ++c) {
      const int i = s * cps + c;
      cp_async_wait<STAGES - 2>();
      __syncthreads();
      issue(i + STAGES - 1);
      const uint32_t xs = sbase + (i % STAGES) * ST_BYTES, fs = xs + XS_BYTES;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t af[4];
        {
          const int row = wrow * 16 + (lane & 15), ch = kk * 2 + (lane >> 4);
          ldsm_x4(xs + row * 128 + ((ch ^ (row & 7)) << 4), af);
        }
#pragma unroll
        for (int jp = 0; jp < NT / 2; ++jp) {
          uint32_t bf[4];
          // factor rows: this warp's hi columns [cb, cb + 8RW), then the same columns of the lo block (row RP + cb ..)
          const int nb = (jp < RW / 2 ? 0 : RP - RW * 8) + cb + jp * 16;
          const int n = nb + (lane & 7) + ((lane >> 4) & 1) * 8, ch = kk * 2 + ((lane >> 3) & 1);
          ldsm_x4(fs + n * 128 + ((ch ^ (n & 7)) << 4), bf);
          mma_bf16(acc[jp * 2 + 0], af, bf[0], bf[1]);
          mma_bf16(acc[jp * 2 + 1], af, bf[2], bf[3]);
        }
      }
    }
    // fold the (factor hi, factor lo) partial products
#pragma unroll
    for (int j = 0; j < RW; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] += acc[j + RW][e];
    if (a.mode == 0) {
      // forward (CS == 1): T (fp32) and the per-slice scaled operand for the GEMM's adapter segment
#pragma unroll
      for (int j = 0; j < RW; ++j) {
        const int col = cb + j * 8 + 2 * t;
        if (ok_lo) *reinterpret_cast<float2*>(a.T + static_cast<size_t>(r_lo) * RP + col) = make_float2(acc[j][0], acc[j][1]);
        if (ok_hi) *reinterpret_cast<float2*>(a.T + static_cast<size_t>(r_hi) * RP + col) = make_float2(acc[j][2], acc[j][3]);
        for (int so = 0; so < a.s_out; ++so) {
          const float2 sc = *reinterpret_cast<const float2*>(a.scales + so * RP + col);
          if (ok_lo) emit(a.U + static_cast<size_t>(r_lo) * a.ldu + so * 3 * RP, col, sc.x * acc[j][0], sc.y * acc[j][1]);
          if (ok_hi) emit(a.U + static_cast<size_t>(r_hi) * a.ldu + so * 3 * RP, col, sc.x * acc[j][2], sc.y * acc[j][3]);
        }
      }
    } else {
      if (s == 0) __syncthreads();                 // red[] zero fill (the main loop has at least one barrier anyway)
#pragma unroll
      for (int j = 0; j < RW; ++j) {
        const int col = cb + j * 8 + 2 * t;
        const float2 sc = *reinterpret_cast<const float2*>(a.scales + s * RP + col);
        d[j][0] = fmaf(sc.x, acc[j][0], d[j][0]); d[j][1] = fmaf(sc.y, acc[j][1], d[j][1]);
        d[j][2] = fmaf(sc.x, acc[j][2], d[j][2]); d[j][3] = fmaf(sc.y, acc[j][3], d[j][3]);
        float p0 = acc[j][0] * t_lo[j].x + acc[j][2] * t_hi[j].x;
        float p1 = acc[j][1] * t_lo[j].y + acc[j][3] * t_hi[j].y;
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
          p0 += __shfl_xor_sync(0xffffffffu, p0, o);
          p1 += __shfl_xor_sync(0xffffffffu, p1, o);
        }
        if (g == 0) {
          atomicAdd(&red[s * RP + col], p0);
          atomicAdd(&red[s * RP + col + 1], p1);
        }
      }
    }
  }
  cp_async_wait<0>();

  if (a.mode != 0) {
#pragma unroll
    for (int j = 0; j < RW; ++j) {
      const int col = cb + j * 8 + 2 * t;
      if (ok_lo) emit(a.U + static_cast<size_t>(r_lo) * a.ldu, col, d[j][0], d[j][1]);
      if (ok_hi) emit(a.U + static_cast<size_t>(r_hi) * a.ldu, col, d[j][2], d[j][3]);
    }
    __syncthreads();
    for (int i = tid; i < CS * RP; i += 256) atomicAdd(a.dc + i, red[i]);
  }
}

static int rows_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

// Resident CTAs per SM (RowsCfg::CTAS): 3 at Rp = 16 / 32 (<= 80 registers, 60 / 72 KB each), 2 at Rp = 64 (<= 128
// registers, 96 KB each).  The grid is whole layers of one CTA per SM, so every SM gets the same share of rows at any CTAS.
template <int RT, int CS>
static int rows_launch_t(RowsArgs a, int num_sms, cudaStream_t st) {
  constexpr int smem = RowsCfg<RT>::SMEM, BM = RowsCfg<RT>::BM;
  static bool done = false;
  if (!done) {
    if (cudaFuncSetAttribute(rows_kernel<RT, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -31;
    done = true;
  }
  // the smallest whole number of CTA "layers" (one CTA on every SM) whose even row share fits a BM-row CTA
  if (num_sms <= 0) num_sms = rows_sm_count();
  int layers = (a.M + num_sms * BM - 1) / (num_sms * BM);
  int grid = layers * num_sms;
  a.rows_per_cta = (a.M + grid - 1) / grid;
  grid = (a.M + a.rows_per_cta - 1) / a.rows_per_cta;
  return launch_pdl_f<8>(rows_kernel<RT, CS>, dim3(grid), dim3(256), smem, st, a) == cudaSuccess ? 0 : -32;
}

int rows_launch(const RowsArgs& a, int rp, int cs, int num_sms, cudaStream_t st) {
  if (a.M <= 0 || a.kslice % R_BK != 0 || (rp != 16 && rp != 32 && rp != 64)) return -30;
  if (a.mode == 0 && cs != 1) return -30;
#define CARA_ROWS(RT, CS) if (rp == RT * 8 && cs == CS) return rows_launch_t<RT, CS>(a, num_sms, st);
  CARA_ROWS(2, 1) CARA_ROWS(2, 3) CARA_ROWS(2, 4) CARA_ROWS(4, 1) CARA_ROWS(4, 3) CARA_ROWS(4, 4)
  CARA_ROWS(8, 1) CARA_ROWS(8, 3) CARA_ROWS(8, 4)
#undef CARA_ROWS
  return -30;
}

// ------------------------------------------------------------------------------------ cols_kernel
constexpr int C_BK = 256, C_BM = 32, C_STAGES = 4;

// Rp = 64 (RT = 8): two warps share each 32-column group of X, one per 32-column half of the rank, so a warp holds as
// many accumulators as at Rp = 32 (<= 128 registers: two CTAs per SM) and a CTA covers 128 columns of X.
template <int RT> struct ColsCfg {
  static constexpr int WH = RT > 4 ? 2 : 1;        // warps per 32-column group of X
  static constexpr int RW = RT / WH;               // 8-column rank tiles per warp
  static constexpr int BK = C_BK / WH;             // X columns per CTA
  static constexpr int VSTR = 2 * RT * 16 + 16;    // padded V row pitch (bytes): the hi and lo blocks
  static constexpr int SMEM = C_STAGES * (C_BM * BK * 2 + ((C_BM * VSTR + 127) / 128) * 128);
};

// HL = 2: V = (hi | lo) column blocks, both contracted; HL = 1: the hi block only (see cols_launch)
template <int RT, int HL>
__global__ void __launch_bounds__(256, RT > 4 ? 2 : 0)     // 0: no minimum, the compiler's own register budget
cols_kernel(const ColsArgs a) {
  using Cfg = ColsCfg<RT>;
  constexpr int RP = RT * 8;
  constexpr int WH = Cfg::WH, RW = Cfg::RW, BK = Cfg::BK;
  constexpr int NT = HL * RW;                      // n-tiles of this warp
  constexpr int NV = HL * RT;                      // 16-byte V chunks per row in shared memory
  constexpr int XCH = BK / 8, XSH = WH == 1 ? 5 : 4;   // 16-byte X chunks per row = 1 << XSH
  constexpr int VSTR = Cfg::VSTR;
  constexpr int XS_BYTES = C_BM * BK * 2;          // 16 KB (8 KB at Rp = 64)
  constexpr int VS_BYTES = C_BM * VSTR;
  constexpr int ST_BYTES = XS_BYTES + ((VS_BYTES + 127) / 128) * 128;
  extern __shared__ __align__(128) uint8_t smem[];
  pdl_wait();
  pdl_trigger();
  const uint32_t sbase = s_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kg = WH == 1 ? warp : (warp & 3);      // this warp's 32-column group of X
  const int half = WH == 1 ? 0 : (warp >> 2);      // and its half of the rank
  const int k0 = blockIdx.x * BK;
  const int slice = k0 / a.slice_w;
  const int m_begin = blockIdx.y * a.rows_per_cta;
  int m_end = m_begin + a.rows_per_cta;
  if (m_end > a.M) m_end = a.M;
  const int nst = (m_end - m_begin + C_BM - 1) / C_BM;

  auto issue = [&](int i) {
    if (i < nst) {
      const uint32_t xs = sbase + (i % C_STAGES) * ST_BYTES, vs = xs + XS_BYTES;
      const int mrow0 = m_begin + i * C_BM;
#pragma unroll
      for (int j = 0; j < C_BM * XCH / 256; ++j) {
        const int idx = j * 256 + tid, row = idx >> XSH, ch = idx & (XCH - 1);
        const bool ok = (mrow0 + row) < m_end;
        const __nv_bfloat16* src = a.X + static_cast<size_t>(ok ? mrow0 + row : 0) * a.ldx + k0 + ch * 8;
        cp_async16(xs + row * (BK * 2) + ((ch ^ (row & 7)) << 4), src, ok);
      }
#pragma unroll
      for (int j = 0; j < (C_BM * NV + 255) / 256; ++j) {
        const int idx = j * 256 + tid;
        if (idx < C_BM * NV) {
          const int row = idx / NV, ch = idx % NV;
          const bool ok = (mrow0 + row) < m_end;
          const __nv_bfloat16* src = a.V + static_cast<size_t>(ok ? mrow0 + row : 0) * a.ldv + slice * 3 * RP + ch * 8;
          cp_async16(vs + row * VSTR + ch * 16, src, ok);
        }
      }
    }
    cp_async_commit();
  };

  float acc[2][NT + 1][4];
#pragma unroll
  for (int kt = 0; kt < 2; ++kt)
#pragma unroll
    for (int j = 0; j <= NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[kt][j][e] = 0.f;
  const uint32_t ones = (lane >> 2) == 0 ? 0x3F803F80u : 0u;   // B fragment of a column of ones (n = 0)

  for (int i = 0; i < C_STAGES - 1; ++i) issue(i);
  for (int i = 0; i < nst; ++i) {
    cp_async_wait<C_STAGES - 2>();
    __syncthreads();
    issue(i + C_STAGES - 1);
    const uint32_t xs = sbase + (i % C_STAGES) * ST_BYTES, vs = xs + XS_BYTES;
#pragma unroll
    for (int ms = 0; ms < C_BM; ms += 16) {
      uint32_t bf[NT / 2][4];
      const int q = lane >> 3;
#pragma unroll
      for (int jp = 0; jp < NT / 2; ++jp) {
        // V tiles: this warp's hi columns [8 RW half, +8 RW), then (HL = 2) the same columns of the lo block
        const int jt = (jp < RW / 2 ? 0 : RT - RW) + half * RW + jp * 2;
        const int row = ms + (lane & 7) + (q & 1) * 8, ch = jt + (q >> 1);
        ldsm_x4_t(vs + row * VSTR + ch * 16, bf[jp]);
      }
#pragma unroll
      for (int kt = 0; kt < 2; ++kt) {
        uint32_t af[4];
        const int row = ms + (lane & 7) + (q >> 1) * 8, ch = (kg * 32 + kt * 16) / 8 + (q & 1);
        ldsm_x4_t(xs + row * (BK * 2) + ((ch ^ (row & 7)) << 4), af);
#pragma unroll
        for (int jp = 0; jp < NT / 2; ++jp) {
          mma_bf16(acc[kt][jp * 2 + 0], af, bf[jp][0], bf[jp][1]);
          mma_bf16(acc[kt][jp * 2 + 1], af, bf[jp][2], bf[jp][3]);
        }
        if (a.colsum != nullptr && half == 0) mma_bf16(acc[kt][NT], af, ones, ones);
      }
    }
  }
  cp_async_wait<0>();

  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int kt = 0; kt < 2; ++kt) {
    const int kc = k0 + kg * 32 + kt * 16 + g;              // X column (output row) of c0/c1; +8 for c2/c3
    if (kc < a.Kc) {
      const int orow = kc - slice * a.slice_w;
#pragma unroll
      for (int j = 0; j < RW; ++j) {
        const int col = half * RW * 8 + j * 8 + 2 * t;
        // 64-bit vector reductions (sm_90+): half as many atomics in the tail every CTA reaches at the same time
        constexpr int LO = (HL - 1) * RW;          // HL = 1: acc[j + LO] is acc[j] itself, counted once below
        const float f = HL == 2 ? 1.0f : 0.5f;
        atomicAdd(reinterpret_cast<float2*>(a.out + static_cast<size_t>(orow) * RP + col),
                  make_float2(f * (acc[kt][j][0] + acc[kt][j + LO][0]), f * (acc[kt][j][1] + acc[kt][j + LO][1])));
        atomicAdd(reinterpret_cast<float2*>(a.out + static_cast<size_t>(orow + 8) * RP + col),
                  make_float2(f * (acc[kt][j][2] + acc[kt][j + LO][2]), f * (acc[kt][j][3] + acc[kt][j + LO][3])));
      }
      if (a.colsum != nullptr && half == 0 && t == 0) {
        atomicAdd(a.colsum + kc, acc[kt][NT][0]);
        atomicAdd(a.colsum + kc + 8, acc[kt][NT][2]);
      }
    }
  }
}

// Resident CTAs per SM: 2 for every (RT, HL) -- <= 128 registers (cols_kernel<8, *> by its launch bounds), 4 x 18.5 /
// 20.5 / 16.5 KB of shared memory at Rp = 16 / 32 / 64 -- which is the `mult` the grid below assumes.
template <int RT, int HL>
static int cols_launch_t(ColsArgs a, int num_sms, cudaStream_t st) {
  constexpr int smem = ColsCfg<RT>::SMEM;
  static bool done = false;
  if (!done) {
    if (cudaFuncSetAttribute(cols_kernel<RT, HL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -41;
    done = true;
  }
  // Exactly `mult` CTAs per SM or fewer, never one more: every SM streams at the same rate, so an SM that gets an
  // extra CTA finishes (mult+1)/mult later and the whole HBM-bound launch waits for it (ncu: 34 % SM-idle at 300 CTAs).
  const int ksplits = a.Kc / ColsCfg<RT>::BK;
  static int mult = -1;
  if (mult < 0) { const char* e = getenv("CARA_COLS_MULT"); mult = (e != nullptr && atoi(e) > 0) ? atoi(e) : 2; }
  int msplits = (mult * num_sms) / ksplits;
  if (msplits < 1) msplits = 1;
  int rows = (a.M + msplits - 1) / msplits;
  rows = ((rows + C_BM - 1) / C_BM) * C_BM;
  msplits = (a.M + rows - 1) / rows;
  a.rows_per_cta = rows;
  return launch_pdl_f<8>(cols_kernel<RT, HL>, dim3(ksplits, msplits), dim3(256), smem, st, a) == cudaSuccess ? 0 : -42;
}

int cols_launch(const ColsArgs& a, int rp, int num_sms, cudaStream_t st) {
  if (a.M <= 0 || a.Kc % C_BK != 0 || a.slice_w % C_BK != 0 || a.Kc % a.slice_w != 0) return -40;
  if (num_sms <= 0) num_sms = 148;
  // CARA_COLS_HL=1 (experiment) contracts only the hi block of V: the sums run over M tokens, so the dropped 2^-9
  // relative lo parts average out (ViT-B worst gradient cosine 0.999942 against 0.999956), for +2.5 % on ViT-L r32 and
  // ~0 on ViT-B r16; the default keeps both blocks.
  static int hl = -1;
  if (hl < 0) { const char* e = getenv("CARA_COLS_HL"); hl = (e != nullptr && e[0] == '1') ? 1 : 2; }
  if (rp == 16) return hl == 2 ? cols_launch_t<2, 2>(a, num_sms, st) : cols_launch_t<2, 1>(a, num_sms, st);
  if (rp == 32) return hl == 2 ? cols_launch_t<4, 2>(a, num_sms, st) : cols_launch_t<4, 1>(a, num_sms, st);
  if (rp == 64) return hl == 2 ? cols_launch_t<8, 2>(a, num_sms, st) : cols_launch_t<8, 1>(a, num_sms, st);
  return -40;
}

}  // namespace cara
