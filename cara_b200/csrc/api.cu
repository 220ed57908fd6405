// C-ABI entry points (include/cara_b200.h).  Thin: validate, translate, launch.
#include "../../include/cara_b200.h"
#include "gemm_sm100.h"
#include "kernels.h"

#include <cstdio>
#include <cstring>

namespace {
thread_local char g_err[512] = "";
thread_local int g_device = -1;

int fail(int code, const char* what) {
  std::snprintf(g_err, sizeof(g_err), "%s (code %d, cuda: %s)", what, code,
                cudaGetErrorString(cudaPeekAtLastError()));
  return code;
}
}  // namespace

extern "C" {

int cara_abi_version(void) { return CARA_B200_ABI_VERSION; }
const char* cara_last_error(void) { return g_err; }

int cara_set_device(int device) {
  if (device == g_device) return 0;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(-1, "cudaSetDevice failed");
  g_device = device;
  return 0;
}

int cara_gemm_cp(const cara_gemm_desc* d, void* stream) {
  if (d == nullptr) return fail(-2, "cara_gemm_cp: null descriptor");
  cara::GemmDesc g{};
  g.M = d->M; g.N = d->N; g.K0 = d->K0;
  g.A0 = static_cast<const __nv_bfloat16*>(d->A0); g.lda0 = d->lda0;
  g.B0 = static_cast<const __nv_bfloat16*>(d->B0); g.ldb0 = d->ldb0;
  g.K1 = d->K1; g.ext_slices = d->ext_slices;
  g.A1 = static_cast<const __nv_bfloat16*>(d->A1); g.lda1 = d->lda1;
  g.B1 = static_cast<const __nv_bfloat16*>(d->B1); g.ldb1 = d->ldb1;
  g.bias = d->bias;
  g.out = static_cast<__nv_bfloat16*>(d->out); g.ldo = d->ldo;
  g.out2 = static_cast<__nv_bfloat16*>(d->out2); g.ldo2 = d->ldo2;
  g.aux = static_cast<const __nv_bfloat16*>(d->aux); g.ldaux = d->ldaux;
  g.epi = d->epi; g.num_sms = d->num_sms;
  g.side = d->side; g.side_rp = d->side_rp; g.side_slices = d->side_slices;
  g.P = static_cast<const __nv_bfloat16*>(d->P); g.ldp = d->ldp;
  g.side_scales = d->side_scales; g.side_T = d->side_T;
  g.side_U = static_cast<__nv_bfloat16*>(d->side_U); g.side_ldu = d->side_ldu;
  g.side_dc = d->side_dc; g.sync = static_cast<unsigned*>(d->sync_ws);
  g.aux2 = static_cast<const __nv_bfloat16*>(d->aux2); g.ldaux2 = d->ldaux2;
  g.delta = d->delta; g.seq_n = d->seq_n;
  int rc = cara::gemm_cp_launch(g, static_cast<cudaStream_t>(stream));
  if (rc != 0) return fail(rc, "cara_gemm_cp: launch failed / bad arguments");
  return 0;
}

#define CARA_STREAM(s) static_cast<cudaStream_t>(s)
#define CARA_RET(rc, name) do { int rc_ = (rc); return rc_ == 0 ? 0 : fail(rc_, name); } while (0)
typedef __nv_bfloat16 bf16;

int cara_ln_fwd(const float* x_in, const void* delta, const float* rowscale, int rows_per_sample, float* x_out,
                const float* gamma, const float* beta, void* h, float* mean, float* rstd, int M, int C, float eps,
                int act_fp32, void* stream) {
  cara::LnFwdArgs a{x_in, delta, rowscale, rows_per_sample > 0 ? rows_per_sample : 1, x_out, gamma, beta, h, mean,
                    rstd, M, C, eps, act_fp32};
  CARA_RET(cara::ln_fwd_launch(a, CARA_STREAM(stream)), "cara_ln_fwd");
}
int cara_ln_bwd(const void* dh, const float* x, const float* mean, const float* rstd, const float* gamma,
                const float* dx_in, float* dx_out, void* g_out, const float* rowscale, int rows_per_sample, int M,
                int C, int act_fp32, void* stream) {
  cara::LnBwdArgs a{dh, x, mean, rstd, gamma, dx_in, dx_out, g_out, rowscale,
                    rows_per_sample > 0 ? rows_per_sample : 1, M, C, act_fp32};
  CARA_RET(cara::ln_bwd_launch(a, CARA_STREAM(stream)), "cara_ln_bwd");
}
int cara_ln_rows_supported(int C, int Rp) { return cara::ln_rows_supported(C, Rp); }
int cara_ln_fwd_rows(const float* x_in, const void* delta, const float* rowscale, int rows_per_sample, float* x_out,
                     const float* gamma, const float* beta, void* h, float* mean, float* rstd, int M, int C, float eps,
                     const void* At2, const float* scales, int slices, int Rp, float* T, void* Uhat, void* stream) {
  cara::LnFwdArgs a{x_in, delta, rowscale, rows_per_sample > 0 ? rows_per_sample : 1, x_out, gamma, beta, h, mean,
                    rstd, M, C, eps, 0};
  const int rc = cara::ln_fwd_rows_launch(a, static_cast<const bf16*>(At2), scales, slices, Rp, T, static_cast<bf16*>(Uhat),
                                          CARA_STREAM(stream));
  if (rc == 1) return fail(-22, "cara_ln_fwd_rows: (C, Rp) not covered, see cara_ln_rows_supported");
  CARA_RET(rc, "cara_ln_fwd_rows");
}
int cara_ln_bwd_rows(const void* dh, const float* x, const float* mean, const float* rstd, const float* gamma,
                     const float* dx_in, float* dx_out, void* g_out, const float* rowscale, int rows_per_sample, int M,
                     int C, const void* Bt2, const float* scales, int Rp, const float* T, void* dThat, float* dscales,
                     void* stream) {
  cara::LnBwdArgs a{dh, x, mean, rstd, gamma, dx_in, dx_out, g_out, rowscale,
                    rows_per_sample > 0 ? rows_per_sample : 1, M, C, 0};
  const int rc = cara::ln_bwd_rows_launch(a, static_cast<const bf16*>(Bt2), scales, Rp, T, static_cast<bf16*>(dThat), dscales,
                                          CARA_STREAM(stream));
  if (rc == 1) return fail(-22, "cara_ln_bwd_rows: (C, Rp) not covered, see cara_ln_rows_supported");
  CARA_RET(rc, "cara_ln_bwd_rows");
}
int cara_adapter_rows_fwd(const void* X, long ldx, int M, int K, const void* At, const float* scales, int slices,
                          int Rp, float* T, void* Uhat, void* stream) {
  cara::RowsArgs a{};
  a.X = static_cast<const bf16*>(X); a.ldx = ldx; a.M = M; a.kslice = K;
  a.Ft = static_cast<const bf16*>(At); a.ldf = K; a.scales = scales; a.mode = 0; a.s_out = slices;
  a.T = T; a.U = static_cast<bf16*>(Uhat); a.ldu = static_cast<long>(slices) * 3 * Rp; a.dc = nullptr;
  CARA_RET(cara::rows_launch(a, Rp, 1, 0, CARA_STREAM(stream)), "cara_adapter_rows_fwd");
}
int cara_adapter_rows_bwd(const void* G, long ldg, int M, int N, int slices, const void* Bt, const float* scales,
                          int Rp, const float* T, void* dThat, float* dscales, void* stream) {
  if (slices < 1 || N % slices != 0) return fail(-30, "cara_adapter_rows_bwd: bad slices");
  cara::RowsArgs a{};
  a.X = static_cast<const bf16*>(G); a.ldx = ldg; a.M = M; a.kslice = N / slices;
  a.Ft = static_cast<const bf16*>(Bt); a.ldf = N / slices; a.scales = scales; a.mode = 1; a.s_out = 0;
  a.T = const_cast<float*>(T); a.U = static_cast<bf16*>(dThat); a.ldu = 3 * Rp; a.dc = dscales;
  CARA_RET(cara::rows_launch(a, Rp, slices, 0, CARA_STREAM(stream)), "cara_adapter_rows_bwd");
}
int cara_adapter_cols(const void* X, long ldx, int M, int Kc, const void* V, long ldv, int slices, int Rp, float* out,
                      float* colsum, void* stream) {
  if (slices < 1 || Kc % slices != 0) return fail(-40, "cara_adapter_cols: bad slices");
  cara::ColsArgs a{};
  a.X = static_cast<const bf16*>(X); a.ldx = ldx; a.M = M; a.Kc = Kc;
  a.V = static_cast<const bf16*>(V); a.ldv = ldv; a.slice_w = Kc / slices; a.out = out; a.colsum = colsum;
  CARA_RET(cara::cols_launch(a, Rp, 0, CARA_STREAM(stream)), "cara_adapter_cols");
}
int cara_attn_fwd(const void* qkv, void* o, void* o_lo, float* lse, int B, int N, int H, int D, float scale,
                  void* stream) {
  cara::AttnArgs a{static_cast<const bf16*>(qkv), static_cast<bf16*>(o), static_cast<bf16*>(o_lo), lse, nullptr,
                   nullptr, nullptr, B, N, H, D, scale};
  CARA_RET(cara::attn_fwd_launch(a, CARA_STREAM(stream)), "cara_attn_fwd");
}
int cara_attn_bwd(const void* qkv, const void* o, const void* o_lo, const float* lse, const void* d_o, void* dqkv,
                  float* delta_ws, int B, int N, int H, int D, float scale, void* stream) {
  cara::AttnArgs a{static_cast<const bf16*>(qkv), static_cast<bf16*>(const_cast<void*>(o)),
                   static_cast<bf16*>(const_cast<void*>(o_lo)), const_cast<float*>(lse),
                   static_cast<const bf16*>(d_o), static_cast<bf16*>(dqkv), delta_ws, B, N, H, D, scale};
  if (o == nullptr && (D != 64 || delta_ws == nullptr))
    return fail(-50, "cara_attn_bwd: a precomputed delta (o == NULL) needs D = 64 and delta_ws");
  CARA_RET(cara::attn_bwd_launch(a, CARA_STREAM(stream)), "cara_attn_bwd");
}
int cara_attn_tiled_fwd(const void* qkv, void* o, void* o_lo, float* lse, int B, int N, int H, int D, float scale,
                        void* stream) {
  if (D != 80 || B <= 0 || N <= 0 || H <= 0 || o == nullptr)
    return fail(-50, "cara_attn_tiled_fwd: needs D = 80, B, N, H >= 1 and o");
  cara::AttnArgs a{static_cast<const bf16*>(qkv), static_cast<bf16*>(o), static_cast<bf16*>(o_lo), lse, nullptr,
                   nullptr, nullptr, B, N, H, D, scale};
  CARA_RET(cara::attn_fwd_tiled_launch(a, CARA_STREAM(stream)), "cara_attn_tiled_fwd");
}
int cara_attn_tiled_bwd(const void* qkv, const void* o, const void* o_lo, const float* lse, const void* d_o, void* dqkv,
                        float* delta_ws, int B, int N, int H, int D, float scale, void* stream) {
  if (D != 80 || B <= 0 || N <= 0 || H <= 0)
    return fail(-50, "cara_attn_tiled_bwd: needs D = 80 and B, N, H >= 1");
  if (o == nullptr || o_lo == nullptr || delta_ws == nullptr)
    return fail(-50, "cara_attn_tiled_bwd: needs o, o_lo and delta_ws (delta is computed here, not taken precomputed)");
  cara::AttnArgs a{static_cast<const bf16*>(qkv), static_cast<bf16*>(const_cast<void*>(o)),
                   static_cast<bf16*>(const_cast<void*>(o_lo)), const_cast<float*>(lse),
                   static_cast<const bf16*>(d_o), static_cast<bf16*>(dqkv), delta_ws, B, N, H, D, scale};
  CARA_RET(cara::attn_bwd_tiled_launch(a, CARA_STREAM(stream)), "cara_attn_tiled_bwd");
}
int cara_gelu_f32(const float* dy, const float* x, float* out, long n, void* stream) {
  CARA_RET(cara::gelu_f32_launch(dy, x, out, n, CARA_STREAM(stream)), "cara_gelu_f32");
}
int cara_attn_f32(const float* qkv, float* o, float* lse, const float* d_o, float* dqkv, int B, int N, int H, int D,
                  float scale, void* stream) {
  CARA_RET(cara::attn_f32_launch(qkv, o, lse, d_o, dqkv, B, N, H, D, scale, CARA_STREAM(stream)), "cara_attn_f32");
}
int cara_debug_read(long long* out, int n) { return cara::attn_debug_read(out, n); }
int cara_resize_normalize(const unsigned char* src, int B, int H, int W, const int* xbounds, const int* xk, int xksize,
                          const int* ybounds, const int* yk, int yksize, unsigned char* tmp, float* out,
                          unsigned char* out_u8, int OH, int OW, const float* mean3, const float* std3, void* stream) {
  if (mean3 == nullptr || std3 == nullptr) return fail(-80, "cara_resize_normalize: mean3 / std3 are host pointers to 3 floats");
  CARA_RET(cara::resize_norm_launch(src, B, H, W, xbounds, xk, xksize, ybounds, yk, yksize, tmp, out, out_u8, OH, OW, mean3,
                                    std3, CARA_STREAM(stream)), "cara_resize_normalize");
}
int cara_patchify(const float* img, void* patches, int B, int Cin, int S, int P, int Kp, void* stream) {
  CARA_RET(cara::patchify_launch(img, static_cast<bf16*>(patches), B, Cin, S, P, Kp, CARA_STREAM(stream)), "cara_patchify");
}
int cara_assemble_tokens(const void* pe, const float* cls, const float* pos, float* x, int B, int N, int C,
                         void* stream) {
  CARA_RET(cara::assemble_launch(static_cast<const bf16*>(pe), cls, pos, x, B, N, C, CARA_STREAM(stream)), "cara_assemble_tokens");
}
int cara_factor_operands(const float* F, void* ext, void* t2, long batch, int rows, int R, int Rp, void* stream) {
  CARA_RET(cara::factor_operands_launch(F, static_cast<bf16*>(ext), static_cast<bf16*>(t2), batch, rows, R, Rp,
                                        CARA_STREAM(stream)), "cara_factor_operands");
}
int cara_stage_terms(const cara_stage_desc* d, int backward, void* stream) {
  if (d == nullptr) return fail(-71, "cara_stage_terms: null descriptor");
  cara::StageArgs a{};
  a.R = d->R; a.Rp = d->Rp; a.C = d->C; a.D = d->D; a.L = d->L;
  a.A1 = d->A1; a.A3 = d->A3; a.A4 = d->A4; a.P1 = d->P1; a.P2 = d->P2; a.R1 = d->R1; a.R2 = d->R2;
  a.bias1 = d->bias1; a.bias2 = d->bias2; a.bias3 = d->bias3;
  a.ai = d->ai; a.pi = d->pi; a.mi = d->mi; a.s_a = d->s_a; a.s_m = d->s_m;
  a.fb_proj = d->fb_proj; a.fb_fc1 = d->fb_fc1; a.fb_fc2 = d->fb_fc2;
  a.kr = d->kr; a.cs_qkv = d->cs_qkv; a.cs_proj = d->cs_proj; a.cs_fc1 = d->cs_fc1; a.a_fc2 = d->a_fc2; a.cs_fc2 = d->cs_fc2;
  a.b_proj = d->b_proj; a.b_fc1 = d->b_fc1; a.b_fc2 = d->b_fc2;
  a.cs_qkv_pad = d->cs_qkv_pad; a.cs_proj_pad = d->cs_proj_pad; a.cs_fc1_pad = d->cs_fc1_pad; a.cs_fc2_pad = d->cs_fc2_pad;
  a.g_kr = d->g_kr; a.g_cs_qkv = d->g_cs_qkv; a.g_cs_proj = d->g_cs_proj; a.g_cs_fc1 = d->g_cs_fc1; a.g_a_fc2 = d->g_a_fc2;
  a.g_cs_fc2 = d->g_cs_fc2; a.g_b_proj = d->g_b_proj; a.g_b_fc1 = d->g_b_fc1; a.g_b_fc2 = d->g_b_fc2;
  a.ld_kr = d->ld_kr; a.ld_cs_qkv = d->ld_cs_qkv; a.ld_cs_proj = d->ld_cs_proj; a.ld_cs_fc1 = d->ld_cs_fc1;
  a.ld_a_fc2 = d->ld_a_fc2; a.ld_cs_fc2 = d->ld_cs_fc2;
  a.dA1 = d->dA1; a.dA3 = d->dA3; a.dA4 = d->dA4; a.dP1 = d->dP1; a.dP2 = d->dP2; a.dR1 = d->dR1; a.dR2 = d->dR2;
  a.dbias1 = d->dbias1; a.dbias2 = d->dbias2; a.dbias3 = d->dbias3;
  CARA_RET(cara::stage_launch(a, backward, CARA_STREAM(stream)), "cara_stage_terms");
}
int cara_merge_weights(const float* W, const float* A, const float* Bf, const float* cs, void* Weff, int N, int K,
                       int slices, int R, void* stream) {
  CARA_RET(cara::merge_launch(W, A, Bf, cs, static_cast<bf16*>(Weff), N, K, slices, R, CARA_STREAM(stream)), "cara_merge_weights");
}
int cara_adamw_step(float* p, const float* g, float* m, float* v, long n, float lr, float beta1, float beta2,
                    float eps, float weight_decay, int step, float gscale, void* stream) {
  CARA_RET(cara::adamw_launch(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, step, gscale, CARA_STREAM(stream)), "cara_adamw_step");
}
int cara_adamw_step_dev(float* p, const float* g, float* m, float* v, long n, float* state, float beta1, float beta2,
                        float eps, float weight_decay, float gscale, void* stream) {
  CARA_RET(cara::adamw_dev_launch(p, g, m, v, n, state, beta1, beta2, eps, weight_decay, gscale, CARA_STREAM(stream)),
           "cara_adamw_step_dev");
}
int cara_sgemm(const float* A, long ars, long acs, const float* B, long brs, long bcs, float* C, long ldc,
               const float* bias, int M, int N, int K, float alpha, float beta, float* workspace, long workspace_floats,
               void* stream) {
  CARA_RET(cara::sgemm_launch(A, ars, acs, B, brs, bcs, C, ldc, bias, M, N, K, alpha, beta, workspace, workspace_floats,
                              CARA_STREAM(stream)), "cara_sgemm");
}

}  // extern "C"
