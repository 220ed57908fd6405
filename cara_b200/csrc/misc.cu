// Small kernels around the hot path: patch embedding staging (timm PatchEmbed as an im2col + GEMM),
// token assembly (cls token + position embedding), eval-mode merge of the CP delta into the frozen
// weights (SURVEY A.3), fused AdamW over one flat fp32 buffer (vit_cp.py:185), and a plain fp32 SIMT
// GEMM for the tiny trainable head (vit_cp.py:166).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "kernels.h"

namespace cara {

// ---------------------------------------------------------------- patchify (im2col for conv PxP / stride P)
// img fp32 [B, Cin, S, S] -> patches bf16 [B*np, Kp], column = (c, py, px), zero padded to Kp.
__global__ void patchify_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out, int B, int Cin,
                                int S, int P, int Kp) {
  const int gp = S / P;
  const long rows = static_cast<long>(B) * gp * gp;
  const int segs = Cin * P;                       // (c, py) segments of P contiguous pixels
  const long total = rows * (segs + 1);           // +1: the zero padding segment
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long row = i / (segs + 1);
    const int seg = static_cast<int>(i % (segs + 1));
    __nv_bfloat16* o = out + row * Kp;
    if (seg == segs) {
      for (int k = segs * P; k < Kp; ++k) o[k] = __float2bfloat16_rn(0.f);
      continue;
    }
    const int b = static_cast<int>(row / (gp * gp)), pi = static_cast<int>(row % (gp * gp));
    const int py0 = (pi / gp) * P, px0 = (pi % gp) * P;
    const int c = seg / P, py = seg % P;
    const float* src = img + ((static_cast<long>(b) * Cin + c) * S + (py0 + py)) * S + px0;
    for (int px = 0; px < P; ++px) o[seg * P + px] = __float2bfloat16_rn(src[px]);
  }
}

// P = 16 (ViT-B/L): one thread per 16-pixel image-row segment, indexed in image memory order, so the fp32 image is
// read as one linear 128-bit stream and every thread writes one aligned 32-byte piece of its patch row
// (the scalar kernel above visited every 128-byte line 16 times: 293 us at batch 256 against a 36 us HBM floor).
__global__ void __launch_bounds__(256)
patchify16_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out, long total, int Cin, int S, int Kp) {
  pdl_wait();
  pdl_trigger();
  const int gp = S / 16;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int pxp = static_cast<int>(i % gp);
    long r = i / gp;
    const int y = static_cast<int>(r % S);
    r /= S;
    const int c = static_cast<int>(r % Cin);
    const long b = r / Cin;
    const float4* src = reinterpret_cast<const float4*>(img + i * 16);
    const float4 v0 = __ldg(src), v1 = __ldg(src + 1), v2 = __ldg(src + 2), v3 = __ldg(src + 3);
    __nv_bfloat162 w[8] = {__floats2bfloat162_rn(v0.x, v0.y), __floats2bfloat162_rn(v0.z, v0.w),
                           __floats2bfloat162_rn(v1.x, v1.y), __floats2bfloat162_rn(v1.z, v1.w),
                           __floats2bfloat162_rn(v2.x, v2.y), __floats2bfloat162_rn(v2.z, v2.w),
                           __floats2bfloat162_rn(v3.x, v3.y), __floats2bfloat162_rn(v3.z, v3.w)};
    const long row = (b * gp + (y >> 4)) * gp + pxp;
    uint4* dst = reinterpret_cast<uint4*>(out + row * Kp + c * 256 + (y & 15) * 16);
    const uint4* wv = reinterpret_cast<const uint4*>(w);
    dst[0] = wv[0];
    dst[1] = wv[1];
  }
}

// x[b, 0, :] = cls + pos[0];  x[b, 1+p, :] = pe[b*np + p, :] + pos[1+p]   (fp32 residual stream)
__global__ void assemble_kernel(const __nv_bfloat16* __restrict__ pe, const float* __restrict__ cls,
                                const float* __restrict__ pos, float* __restrict__ x, int B, int N, int C) {
  pdl_wait();
  pdl_trigger();
  const long total = static_cast<long>(B) * N * (C / 4);
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % (C / 4));
    const long tok = i / (C / 4);
    const int n = static_cast<int>(tok % N), b = static_cast<int>(tok / N);
    const float4 p = *reinterpret_cast<const float4*>(pos + static_cast<long>(n) * C + c4 * 4);
    float4 v;
    if (n == 0) {
      v = *reinterpret_cast<const float4*>(cls + c4 * 4);
    } else {
      const uint2 u = *reinterpret_cast<const uint2*>(pe + (static_cast<long>(b) * (N - 1) + (n - 1)) * C + c4 * 4);
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
      const float2 d = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
      v = make_float4(a.x, a.y, d.x, d.y);
    }
    v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
    *reinterpret_cast<float4*>(x + tok * C + c4 * 4) = v;
  }
}

int patchify_launch(const float* img, __nv_bfloat16* out, int B, int Cin, int S, int P, int Kp, cudaStream_t st) {
  if (S % P != 0 || Kp < Cin * P * P) return -60;
  if (P == 16 && Kp == Cin * 256 && (reinterpret_cast<uintptr_t>(img) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    const long total = static_cast<long>(B) * Cin * S * (S / 16);
    return launch_pdl_f<16>(patchify16_kernel, dim3(148 * 16), dim3(256), 0, st, img, out, total, Cin, S, Kp) == cudaSuccess ? 0 : -61;
  }
  patchify_kernel<<<148 * 8, 256, 0, st>>>(img, out, B, Cin, S, P, Kp);
  return cudaGetLastError() == cudaSuccess ? 0 : -61;
}
int assemble_launch(const __nv_bfloat16* pe, const float* cls, const float* pos, float* x, int B, int N, int C,
                    cudaStream_t st) {
  if (C % 4 != 0) return -62;
  return launch_pdl_f<16>(assemble_kernel, dim3(148 * 8), dim3(256), 0, st, pe, cls, pos, x, B, N, C) == cudaSuccess ? 0 : -63;
}

// ---------------------------------------------------------------- staged factor operands
// F fp32 [batch, rows, R] -> ext bf16 [batch, rows, 3Rp] = [hi | hi | lo] (adapter segment of the GEMM) and
// t2 bf16 [batch, 2Rp, rows] = [hi^T ; lo^T] (skinny kernels), hi + lo ~ F to ~16 mantissa bits, zero padded to Rp.
// One launch per factor instead of the ~10 elementwise / cat / transpose kernels of the torch formulation.
__global__ void __launch_bounds__(256)
factor_operands_kernel(const float* __restrict__ F, __nv_bfloat16* __restrict__ ext, __nv_bfloat16* __restrict__ t2,
                       long total, int rows, int R, int Rp) {
  for (long i = blockIdx.x * 256L + threadIdx.x; i < total; i += gridDim.x * 256L) {
    const int r = static_cast<int>(i % Rp);
    const long br = i / Rp;                       // batch * rows + row
    const int row = static_cast<int>(br % rows);
    const long b = br / rows;
    const float v = r < R ? F[br * R + r] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    __nv_bfloat16* e = ext + br * 3 * Rp;
    e[r] = hi; e[Rp + r] = hi; e[2 * Rp + r] = lo;
    __nv_bfloat16* t = t2 + b * 2 * Rp * rows;
    t[static_cast<long>(r) * rows + row] = hi;
    t[static_cast<long>(Rp + r) * rows + row] = lo;
  }
}
int factor_operands_launch(const float* F, __nv_bfloat16* ext, __nv_bfloat16* t2, long batch, int rows, int R, int Rp,
                           cudaStream_t st) {
  if (batch <= 0 || rows <= 0 || R <= 0 || Rp < R) return -64;
  const long total = batch * rows * Rp;
  long grid = (total + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  factor_operands_kernel<<<static_cast<int>(grid), 256, 0, st>>>(F, ext, t2, total, rows, R, Rp);
  return cudaGetLastError() == cudaSuccess ? 0 : -65;
}

// ---------------------------------------------------------------- per-step staging of the CP factors (SURVEY A.1 / A.2)
// The twelve CP_* parameters of the root model (cara.py:112-125) -> the per-layer, per-projection terms the kernels
// consume, and the chain rule back (SURVEY A.2 "chain to parameters").  One launch each way instead of ~90 tiny torch
// kernels per step.  All tensors fp32; R = rank, Rp = rank padded to 16 / 32 (the padded copies of the cs terms are what
// the kernels read; they carry no gradient).
//   kr[h*D+d, r]        = A3[h,r] A4[d,r]                          (out-side factor of qkv: Khatri-Rao of CP_A3, CP_A4)
//   cs_qkv[l,k,r]       = s_a[l] R1[r] A1[ai[l]+k, r]              (cara.py:26: rows attn_idx .. attn_idx+2)
//   cs_proj[l,r]        = s_a[l] R2[r] P1[pi[l], r]                (cara.py:51)
//   cs_fc1[l,a,r]       = s_m[l] R2[r] P1[mi[l]+a, r]              (cara.py:72)
//   a_fc2[l, a*C+b, r]  = P1[mi[l]+4+a, r] P2[b,r]                 (cara.py:73: in-side factor of fc2)
//   cs_fc2[l,r]         = s_m[l] R2[r]
//   b_proj[l,c] = fb_proj[l,c] + s_a[l] bias1[c];  b_fc1[l,c] = fb_fc1[l,c] + s_m[l] bias2[c];  b_fc2 likewise with bias3
__global__ void __launch_bounds__(256)
stage_fwd_kernel(const StageArgs a) {
  const int R = a.R, Rp = a.Rp, C = a.C, D = a.D, L = a.L;
  const long n_kr = static_cast<long>(C) * R, n_q = static_cast<long>(L) * 3 * R, n_p = static_cast<long>(L) * R,
             n_1 = static_cast<long>(L) * 4 * R, n_a = static_cast<long>(L) * 4 * C * R, n_bp = static_cast<long>(L) * C,
             n_b1 = static_cast<long>(L) * 4 * C;
  const long total = n_kr + n_q + n_p + n_1 + n_a + n_p + n_bp + n_b1 + n_bp;
  for (long i = blockIdx.x * 256L + threadIdx.x; i < total; i += gridDim.x * 256L) {
    long j = i;
    if (j < n_kr) {
      const int r = static_cast<int>(j % R), row = static_cast<int>(j / R);
      a.kr[j] = a.A3[(row / D) * R + r] * a.A4[(row % D) * R + r];
      continue;
    }
    j -= n_kr;
    if (j < n_q) {
      const int r = static_cast<int>(j % R), k = static_cast<int>((j / R) % 3), l = static_cast<int>(j / (3 * R));
      const float v = a.s_a[l] * a.R1[r] * a.A1[static_cast<long>(a.ai[l] + k) * R + r];
      a.cs_qkv[j] = v;
      a.cs_qkv_pad[(static_cast<long>(l) * 3 + k) * Rp + r] = v;
      continue;
    }
    j -= n_q;
    if (j < n_p) {
      const int r = static_cast<int>(j % R), l = static_cast<int>(j / R);
      const float v = a.s_a[l] * a.R2[r] * a.P1[static_cast<long>(a.pi[l]) * R + r];
      a.cs_proj[j] = v;
      a.cs_proj_pad[static_cast<long>(l) * Rp + r] = v;
      continue;
    }
    j -= n_p;
    if (j < n_1) {
      const int r = static_cast<int>(j % R), k = static_cast<int>((j / R) % 4), l = static_cast<int>(j / (4 * R));
      const float v = a.s_m[l] * a.R2[r] * a.P1[static_cast<long>(a.mi[l] + k) * R + r];
      a.cs_fc1[j] = v;
      a.cs_fc1_pad[(static_cast<long>(l) * 4 + k) * Rp + r] = v;
      continue;
    }
    j -= n_1;
    if (j < n_a) {
      const int r = static_cast<int>(j % R);
      const long row = j / R;                                    // l * 4C + k * C + b
      const int bcol = static_cast<int>(row % C), k = static_cast<int>((row / C) % 4), l = static_cast<int>(row / (4L * C));
      a.a_fc2[j] = a.P1[static_cast<long>(a.mi[l] + 4 + k) * R + r] * a.P2[static_cast<long>(bcol) * R + r];
      continue;
    }
    j -= n_a;
    if (j < n_p) {
      const int r = static_cast<int>(j % R), l = static_cast<int>(j / R);
      const float v = a.s_m[l] * a.R2[r];
      a.cs_fc2[j] = v;
      a.cs_fc2_pad[static_cast<long>(l) * Rp + r] = v;
      continue;
    }
    j -= n_p;
    if (j < n_bp) { a.b_proj[j] = a.fb_proj[j] + a.s_a[j / C] * a.bias1[j % C]; continue; }
    j -= n_bp;
    if (j < n_b1) { a.b_fc1[j] = a.fb_fc1[j] + a.s_m[j / (4 * C)] * a.bias2[j % (4 * C)]; continue; }
    j -= n_b1;
    a.b_fc2[j] = a.fb_fc2[j] + a.s_m[j / C] * a.bias3[j % C];
  }
}

// Chain rule of the staging above: gradients of the nine staged tensors (any may be null; the R-wide ones come with a
// row pitch, they are views into the Rp-wide gradient sink) -> gradients of CP_A1, CP_A3, CP_A4, CP_P1, CP_P2 (its
// a_fc2 share), CP_R1, CP_R2, CP_bias1..3.  One thread per output element, serial reductions (at most C terms);
// the indexed rows are added atomically into zero-filled outputs (rows are distinct for every model set_cara builds).
__global__ void __launch_bounds__(256)
stage_bwd_kernel(const StageArgs a) {
  const int R = a.R, C = a.C, D = a.D, H = C / a.D, L = a.L;
  const long n_q = static_cast<long>(L) * 3 * R, n_3 = static_cast<long>(H) * R, n_4 = static_cast<long>(D) * R,
             n_p = static_cast<long>(L) * R, n_1 = static_cast<long>(L) * 4 * R, n_2 = static_cast<long>(C) * R;
  const long total = n_q + R + n_3 + n_4 + n_p + n_1 + n_1 + n_2 + R + 6L * C;
  for (long i = blockIdx.x * 256L + threadIdx.x; i < total; i += gridDim.x * 256L) {
    long j = i;
    if (j < n_q) {                                               // dCP_A1[ai[l]+k] += s_a dcs_qkv[l,k] (.) R1
      if (a.g_cs_qkv != nullptr) {
        const int r = static_cast<int>(j % R), k = static_cast<int>((j / R) % 3), l = static_cast<int>(j / (3 * R));
        atomicAdd(a.dA1 + static_cast<long>(a.ai[l] + k) * R + r,
                  a.s_a[l] * a.g_cs_qkv[(static_cast<long>(l) * 3 + k) * a.ld_cs_qkv + r] * a.R1[r]);
      }
      continue;
    }
    j -= n_q;
    if (j < R) {                                                 // dCP_R1 = sum_{l,k} s_a dcs_qkv[l,k] (.) A1[ai[l]+k]
      if (a.g_cs_qkv != nullptr) {
        const int r = static_cast<int>(j);
        float acc = 0.f;
        for (int l = 0; l < L; ++l)
          for (int k = 0; k < 3; ++k)
            acc = fmaf(a.s_a[l] * a.g_cs_qkv[(static_cast<long>(l) * 3 + k) * a.ld_cs_qkv + r],
                       a.A1[static_cast<long>(a.ai[l] + k) * R + r], acc);
        a.dR1[r] = acc;
      }
      continue;
    }
    j -= R;
    if (j < n_3) {                                               // dCP_A3[h] = sum_d dKR[h,d] (.) A4[d]
      if (a.g_kr != nullptr) {
        const int r = static_cast<int>(j % R), h = static_cast<int>(j / R);
        float acc = 0.f;
        for (int d = 0; d < D; ++d) acc = fmaf(a.g_kr[static_cast<long>(h * D + d) * a.ld_kr + r], a.A4[d * R + r], acc);
        a.dA3[j] = acc;
      }
      continue;
    }
    j -= n_3;
    if (j < n_4) {                                               // dCP_A4[d] = sum_h dKR[h,d] (.) A3[h]
      if (a.g_kr != nullptr) {
        const int r = static_cast<int>(j % R), d = static_cast<int>(j / R);
        float acc = 0.f;
        for (int h = 0; h < H; ++h) acc = fmaf(a.g_kr[static_cast<long>(h * D + d) * a.ld_kr + r], a.A3[h * R + r], acc);
        a.dA4[j] = acc;
      }
      continue;
    }
    j -= n_4;
    if (j < n_p) {                                               // dCP_P1[pi[l]] += s_a dcs_proj[l] (.) R2
      if (a.g_cs_proj != nullptr) {
        const int r = static_cast<int>(j % R), l = static_cast<int>(j / R);
        atomicAdd(a.dP1 + static_cast<long>(a.pi[l]) * R + r, a.s_a[l] * a.g_cs_proj[static_cast<long>(l) * a.ld_cs_proj + r] * a.R2[r]);
      }
      continue;
    }
    j -= n_p;
    if (j < n_1) {                                               // dCP_P1[mi[l]+k] += s_m dcs_fc1[l,k] (.) R2
      if (a.g_cs_fc1 != nullptr) {
        const int r = static_cast<int>(j % R), k = static_cast<int>((j / R) % 4), l = static_cast<int>(j / (4 * R));
        atomicAdd(a.dP1 + static_cast<long>(a.mi[l] + k) * R + r,
                  a.s_m[l] * a.g_cs_fc1[(static_cast<long>(l) * 4 + k) * a.ld_cs_fc1 + r] * a.R2[r]);
      }
      continue;
    }
    j -= n_1;
    if (j < n_1) {                                               // dCP_P1[mi[l]+4+k] += sum_b dA_fc2[l,k,b] (.) P2[b]
      if (a.g_a_fc2 != nullptr) {
        const int r = static_cast<int>(j % R), k = static_cast<int>((j / R) % 4), l = static_cast<int>(j / (4 * R));
        const float* g = a.g_a_fc2 + (static_cast<long>(l) * 4 + k) * C * a.ld_a_fc2 + r;
        float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
        int bcol = 0;
        for (; bcol + 3 < C; bcol += 4) {
          acc0 = fmaf(g[static_cast<long>(bcol) * a.ld_a_fc2], a.P2[static_cast<long>(bcol) * R + r], acc0);
          acc1 = fmaf(g[static_cast<long>(bcol + 1) * a.ld_a_fc2], a.P2[static_cast<long>(bcol + 1) * R + r], acc1);
          acc2 = fmaf(g[static_cast<long>(bcol + 2) * a.ld_a_fc2], a.P2[static_cast<long>(bcol + 2) * R + r], acc2);
          acc3 = fmaf(g[static_cast<long>(bcol + 3) * a.ld_a_fc2], a.P2[static_cast<long>(bcol + 3) * R + r], acc3);
        }
        for (; bcol < C; ++bcol) acc0 = fmaf(g[static_cast<long>(bcol) * a.ld_a_fc2], a.P2[static_cast<long>(bcol) * R + r], acc0);
        atomicAdd(a.dP1 + static_cast<long>(a.mi[l] + 4 + k) * R + r, (acc0 + acc1) + (acc2 + acc3));
      }
      continue;
    }
    j -= n_1;
    if (j < n_2) {                                               // dCP_P2[b] (a_fc2 share) = sum_{l,k} dA_fc2[l,k,b] (.) P1[mi[l]+4+k]
      if (a.g_a_fc2 != nullptr) {
        const int r = static_cast<int>(j % R), bcol = static_cast<int>(j / R);
        float acc = 0.f;
        for (int l = 0; l < L; ++l)
          for (int k = 0; k < 4; ++k)
            acc = fmaf(a.g_a_fc2[((static_cast<long>(l) * 4 + k) * C + bcol) * a.ld_a_fc2 + r],
                       a.P1[static_cast<long>(a.mi[l] + 4 + k) * R + r], acc);
        a.dP2[j] = acc;
      }
      continue;
    }
    j -= n_2;
    if (j < R) {                                                 // dCP_R2
      const int r = static_cast<int>(j);
      float acc = 0.f;
      for (int l = 0; l < L; ++l) {
        if (a.g_cs_proj != nullptr)
          acc = fmaf(a.s_a[l] * a.g_cs_proj[static_cast<long>(l) * a.ld_cs_proj + r], a.P1[static_cast<long>(a.pi[l]) * R + r], acc);
        if (a.g_cs_fc1 != nullptr)
          for (int k = 0; k < 4; ++k)
            acc = fmaf(a.s_m[l] * a.g_cs_fc1[(static_cast<long>(l) * 4 + k) * a.ld_cs_fc1 + r],
                       a.P1[static_cast<long>(a.mi[l] + k) * R + r], acc);
        if (a.g_cs_fc2 != nullptr) acc = fmaf(a.s_m[l], a.g_cs_fc2[static_cast<long>(l) * a.ld_cs_fc2 + r], acc);
      }
      a.dR2[r] = acc;
      continue;
    }
    j -= R;
    {                                                            // dCP_bias1 [C], dCP_bias2 [4C], dCP_bias3 [C]
      const float* g; const float* sc; float* out; int width; long col;
      if (j < C) { g = a.g_b_proj; sc = a.s_a; out = a.dbias1; width = C; col = j; }
      else if (j < 5L * C) { g = a.g_b_fc1; sc = a.s_m; out = a.dbias2; width = 4 * C; col = j - C; }
      else { g = a.g_b_fc2; sc = a.s_m; out = a.dbias3; width = C; col = j - 5L * C; }
      if (g != nullptr) {
        float acc = 0.f;
        for (int l = 0; l < L; ++l) acc = fmaf(sc[l], g[static_cast<long>(l) * width + col], acc);
        out[col] = acc;
      }
    }
  }
}

int stage_launch(const StageArgs& a, int backward, cudaStream_t st) {
  if (a.R <= 0 || a.Rp < a.R || a.C <= 0 || a.D <= 0 || a.C % a.D != 0 || a.L <= 0) return -71;
  long total;
  if (!backward) total = static_cast<long>(a.C) * a.R * (1 + 4L * a.L) + static_cast<long>(a.L) * (9L * a.R + 6L * a.C);
  else total = static_cast<long>(a.L) * 12 * a.R + 2L * a.R + static_cast<long>(a.C / a.D + a.D + a.C) * a.R + 6L * a.C;
  long grid = (total + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  if (backward) stage_bwd_kernel<<<static_cast<int>(grid), 256, 0, st>>>(a);
  else stage_fwd_kernel<<<static_cast<int>(grid), 256, 0, st>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : -72;
}

// ---------------------------------------------------------------- eval-mode merge (SURVEY A.3)
// Weff[n, k] = W[n, k] + sum_r (Bf[n mod w, r] * cs[n / w, r]) * A[k, r]      W fp32 -> Weff bf16
template <int R>
__global__ void __launch_bounds__(128)
merge_kernel(const float* __restrict__ W, const float* __restrict__ A, const float* __restrict__ Bf,
             const float* __restrict__ cs, __nv_bfloat16* __restrict__ out, int N, int K, int w) {
  __shared__ float bc[8][R];
  const int n0 = blockIdx.y * 8;
  for (int i = threadIdx.x; i < 8 * R; i += 128) {
    const int n = n0 + i / R, r = i % R;
    bc[i / R][r] = n < N ? Bf[static_cast<long>(n % w) * R + r] * cs[(n / w) * R + r] : 0.f;
  }
  __syncthreads();
  const int k = (blockIdx.x * 128 + threadIdx.x) * 2;
  if (k >= K) return;
  float a0[R], a1[R];
#pragma unroll
  for (int r = 0; r < R; ++r) { a0[r] = A[static_cast<long>(k) * R + r]; a1[r] = A[static_cast<long>(k + 1) * R + r]; }
  for (int i = 0; i < 8 && n0 + i < N; ++i) {
    const float2 wv = *reinterpret_cast<const float2*>(W + static_cast<long>(n0 + i) * K + k);
    float d0 = wv.x, d1 = wv.y;
#pragma unroll
    for (int r = 0; r < R; ++r) { d0 = fmaf(bc[i][r], a0[r], d0); d1 = fmaf(bc[i][r], a1[r], d1); }
    *reinterpret_cast<__nv_bfloat162*>(out + static_cast<long>(n0 + i) * K + k) = __floats2bfloat162_rn(d0, d1);
  }
}

int merge_launch(const float* W, const float* A, const float* Bf, const float* cs, __nv_bfloat16* out, int N, int K,
                 int slices, int R, cudaStream_t st) {
  if (K % 2 != 0 || slices < 1 || N % slices != 0) return -64;
  const dim3 grid((K / 2 + 127) / 128, (N + 7) / 8);
  const int w = N / slices;
  switch (R) {
    case 4: merge_kernel<4><<<grid, 128, 0, st>>>(W, A, Bf, cs, out, N, K, w); break;
    case 8: merge_kernel<8><<<grid, 128, 0, st>>>(W, A, Bf, cs, out, N, K, w); break;
    case 16: merge_kernel<16><<<grid, 128, 0, st>>>(W, A, Bf, cs, out, N, K, w); break;
    case 32: merge_kernel<32><<<grid, 128, 0, st>>>(W, A, Bf, cs, out, N, K, w); break;
    case 64: merge_kernel<64><<<grid, 128, 0, st>>>(W, A, Bf, cs, out, N, K, w); break;
    default: return -65;
  }
  return cudaGetLastError() == cudaSuccess ? 0 : -66;
}

// ---------------------------------------------------------------- fused AdamW (torch.optim.AdamW semantics)
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, long n, float lr, float b1, float b2, float eps, float wd,
                             float bc1, float bc2_sqrt, float gscale) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * gscale;
    float pi = p[i] * (1.0f - lr * wd);
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    pi -= (lr / bc1) * mi / denom;
    p[i] = pi; m[i] = mi; v[i] = vi;
  }
}
int adamw_launch(float* p, const float* g, float* m, float* v, long n, float lr, float b1, float b2, float eps,
                 float wd, int step, float gscale, cudaStream_t st) {
  if (n <= 0 || step < 1) return -67;
  const float bc1 = 1.0f - powf(b1, static_cast<float>(step));
  const float bc2s = sqrtf(1.0f - powf(b2, static_cast<float>(step)));
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  adamw_kernel<<<grid, 256, 0, st>>>(p, g, m, v, n, lr, b1, b2, eps, wd, bc1, bc2s, gscale);
  return cudaGetLastError() == cudaSuccess ? 0 : -68;
}

// Same update with the two per-step scalars read from DEVICE memory, so that the launch can sit inside a replayed CUDA
// graph: state[0] = learning rate (written by the host, stream-ordered, whenever the schedule changes it),
// state[1] = number of optimizer steps taken so far (advanced here), state[2] = exit ticket (int bits).
// Every thread reads state[] before its block takes a ticket; the block that takes the last ticket is the only writer.
__global__ void adamw_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                 float* __restrict__ v, long n, float* __restrict__ state, float b1, float b2, float eps,
                                 float wd, float gscale) {
  // bias corrections in double by one thread per block (1 - b2^t for small t loses its digits in fast-math fp32)
  __shared__ float s_hp[4];
  if (threadIdx.x == 0) {
    const float lr0 = *reinterpret_cast<volatile float*>(state);
    const float t = *reinterpret_cast<volatile float*>(state + 1) + 1.0f;
    s_hp[0] = lr0;
    s_hp[1] = t;
    s_hp[2] = static_cast<float>(1.0 - pow(static_cast<double>(b1), static_cast<double>(t)));
    s_hp[3] = static_cast<float>(sqrt(1.0 - pow(static_cast<double>(b2), static_cast<double>(t))));
  }
  __syncthreads();
  const float lr = s_hp[0], step = s_hp[1], bc1 = s_hp[2], bc2_sqrt = s_hp[3];
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * gscale;
    float pi = p[i] * (1.0f - lr * wd);
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    pi -= (lr / bc1) * mi / denom;
    p[i] = pi; m[i] = mi; v[i] = vi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    int* ticket = reinterpret_cast<int*>(state + 2);
    if (atomicAdd(ticket, 1) == static_cast<int>(gridDim.x) - 1) {
      *ticket = 0;
      state[1] = step;
      __threadfence();
    }
  }
}
int adamw_dev_launch(float* p, const float* g, float* m, float* v, long n, float* state, float b1, float b2, float eps,
                     float wd, float gscale, cudaStream_t st) {
  if (n <= 0 || state == nullptr) return -67;
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  adamw_dev_kernel<<<grid, 256, 0, st>>>(p, g, m, v, n, state, b1, b2, eps, wd, gscale);
  return cudaGetLastError() == cudaSuccess ? 0 : -68;
}

// ---------------------------------------------------------------- fp32 SIMT GEMM with general strides
// C[m,n] = alpha * sum_k A(m,k) B(k,n) + beta * C[m,n] + bias[n];  A(m,k) = A[m*ars + k*acs], B(k,n) = B[k*brs + n*bcs]
__global__ void __launch_bounds__(256)
sgemm_kernel(const float* __restrict__ A, long ars, long acs, const float* __restrict__ B, long brs, long bcs,
             float* __restrict__ C, long ldc, const float* __restrict__ bias, int M, int N, int K, float alpha,
             float beta, int kper, float* __restrict__ ws) {
  __shared__ float As[16][65], Bs[16][65];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  // split-K (gridDim.z > 1): this CTA reduces k in [kbeg, kend) into its own slice of the workspace
  const int kbeg = blockIdx.z * kper;
  const int kend = (kbeg + kper < K) ? kbeg + kper : K;
  K = kend;
  float acc[4][4] = {};
  for (int k0 = kbeg; k0 < K; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {
      const int kk = i & 15, r = i >> 4;
      As[kk][r] = (m0 + r < M && k0 + kk < K) ? A[(m0 + r) * ars + (k0 + kk) * acs] : 0.f;
      Bs[kk][r] = (n0 + r < N && k0 + kk < K) ? B[(k0 + kk) * brs + (n0 + r) * bcs] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = alpha * acc[i][j];
      if (gridDim.z > 1) {                      // split-K: partial sums, reduced in a fixed order by sgemm_reduce_kernel
        ws[(static_cast<long>(blockIdx.z) * M + m) * N + n] = v;
        continue;
      }
      if (bias != nullptr) v += bias[n];
      if (beta != 0.f) v += beta * C[m * ldc + n];
      C[m * ldc + n] = v;
    }
  }
}
// C[m,n] = sum_z ws[z,m,n] + bias[n]: the split-K partial sums in a fixed order (no atomics: every run of the same step
// produces the same bits -- fp32 noise in the logits would flip bf16 roundings all the way down the backward pass)
__global__ void __launch_bounds__(256)
sgemm_reduce_kernel(const float* __restrict__ ws, float* __restrict__ C, const float* __restrict__ bias, long MN, int N,
                    int splits) {
  for (long i = blockIdx.x * 256L + threadIdx.x; i < MN; i += gridDim.x * 256L) {
    float v = 0.f;
    for (int z = 0; z < splits; ++z) v += ws[z * MN + i];
    if (bias != nullptr) v += bias[i % N];
    C[i] = v;
  }
}

int sgemm_launch(const float* A, long ars, long acs, const float* B, long brs, long bcs, float* C, long ldc,
                 const float* bias, int M, int N, int K, float alpha, float beta, float* ws, long ws_floats,
                 cudaStream_t st) {
  if (M <= 0 || N <= 0 || K <= 0) return -69;
  const int gx = (N + 63) / 64, gy = (M + 63) / 64;
  // The classifier head's three GEMMs (e.g. 256 x 100 x 768) fill 8-48 CTAs and are pure latency chains over K:
  // split K across ~2 CTAs per SM when C is a plain contiguous output and the caller lent a workspace.
  int splits = 1;
  if (ws != nullptr && beta == 0.f && ldc == N && gx * gy < 74 && K >= 128) {
    splits = (2 * 148) / (gx * gy);
    if (splits > K / 32) splits = K / 32;
    while (splits > 1 && static_cast<long>(splits) * M * N > ws_floats) --splits;
    if (splits < 1) splits = 1;
  }
  int kper = ((K + splits - 1) / splits + 15) / 16 * 16;
  splits = (K + kper - 1) / kper;
  sgemm_kernel<<<dim3(gx, gy, splits), 256, 0, st>>>(A, ars, acs, B, brs, bcs, C, ldc, bias, M, N, K, alpha, beta, kper, ws);
  if (splits > 1) {
    const long MN = static_cast<long>(M) * N;
    long grid = (MN + 255) / 256;
    if (grid > 148 * 4) grid = 148 * 4;
    sgemm_reduce_kernel<<<static_cast<int>(grid), 256, 0, st>>>(ws, C, bias, MN, N, splits);
  }
  return cudaGetLastError() == cudaSuccess ? 0 : -70;
}

}  // namespace cara
