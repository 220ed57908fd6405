// Internal launch interfaces of the non-GEMM kernels.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <stdlib.h>
#include <utility>

namespace cara {

// Programmatic dependent launch (sm_90+), OFF by default (CARA_PDL = bit mask of kernel families, see pdl_mask): every hot kernel can be launched
// with "programmatic stream serialization"; it starts with pdl_wait() -- which returns once the preceding kernel in
// the stream has completed and flushed -- and calls pdl_trigger() right after, so the NEXT kernel's CTAs are already
// resident when this one ends.  Nothing touches global memory before pdl_wait().  Measured on the ViT-B/16 step
// (two A/B pairs on one box): 7,187 / 7,160 img/s with it against 7,367 / 7,338 without -- the early CTAs land on
// whichever SMs drain first, which breaks the even CTAs-per-SM placement the HBM-bound kernels are sized for.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
// pdl_mask bit per kernel family (CARA_PDL is a bit mask: 1 GEMM, 2 attention, 4 LayerNorm, 8 rows/cols, 16 small)
inline int pdl_mask() {
  static int m = -1;
  if (m < 0) { const char* e = getenv("CARA_PDL"); m = e != nullptr ? atoi(e) : 0; }
  return m;
}
template <int FAMILY, typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_f(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_mask() & FAMILY) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(std::forward<Args>(args))...);
}

struct LnFwdArgs {
  const float* x_in; const void* delta; const float* rowscale; int rows_per_sample;
  float* x_out; const float* gamma; const float* beta; void* h; float* mean; float* rstd;
  int M, C; float eps; int act_fp32;
};
struct LnBwdArgs {
  const void* dh; const float* x; const float* mean; const float* rstd; const float* gamma;
  const float* dx_in; float* dx_out; void* g_out; const float* rowscale; int rows_per_sample;
  int M, C; int act_fp32;
};
int ln_fwd_launch(const LnFwdArgs& a, cudaStream_t st);
int ln_bwd_launch(const LnBwdArgs& a, cudaStream_t st);
// ln_rows.cu: the same LayerNorms fused with the rank-R row contraction of the projection they feed (bf16 only).
// 0 = launched, 1 = (C, Rp) not covered, < 0 = error.
int ln_rows_supported(int C, int rp);
int ln_fwd_rows_launch(const LnFwdArgs& l, const __nv_bfloat16* Ft, const float* scales, int slices, int rp, float* T,
                       __nv_bfloat16* U, cudaStream_t st);
int ln_bwd_rows_launch(const LnBwdArgs& l, const __nv_bfloat16* Ft, const float* scales, int rp, const float* T,
                       __nv_bfloat16* dT, float* dc, cudaStream_t st);

// Tall-skinny adapter contractions (skinny.cu)
struct RowsArgs {
  const __nv_bfloat16* X; long ldx; int M; int kslice;  // X [M, CS*kslice]
  const __nv_bfloat16* Ft; long ldf;                     // factor transposed [Rp, kslice]
  const float* scales;                                   // fwd [s_out, Rp] / bwd [CS, Rp]
  int mode;                                              // 0 fwd, 1 bwd
  int s_out;
  float* T;                                              // [M, Rp] fp32 (fwd: out, bwd: in)
  __nv_bfloat16* U; long ldu;                            // fwd Uhat [M, s_out*Rp] / bwd dThat [M, Rp]
  float* dc;                                             // bwd [CS, Rp], atomically accumulated
  int rows_per_cta;                                      // set by rows_launch (<= 128)
};
int rows_launch(const RowsArgs& a, int rp, int cs, int num_sms, cudaStream_t st);

struct ColsArgs {
  const __nv_bfloat16* X; long ldx; int M; int Kc;      // X [M, Kc]
  const __nv_bfloat16* V; long ldv;                      // V [M, (Kc/slice_w)*Rp]
  int slice_w;
  float* out;                                            // [slice_w, Rp] fp32, accumulated
  float* colsum;                                         // [Kc] fp32 or null, accumulated
  int rows_per_cta;
};
int cols_launch(const ColsArgs& a, int rp, int num_sms, cudaStream_t st);

// Attention core (attention.cu): qkv [B, N, 3, H, D] -> o [B, N, H, D]
struct AttnArgs {
  const __nv_bfloat16* qkv; __nv_bfloat16* o; __nv_bfloat16* o_lo; float* lse;   // lse [B, H, N] (log2 domain)
  const __nv_bfloat16* d_o; __nv_bfloat16* dqkv;                // backward only
  float* delta;                                                 // backward workspace [B, H, N] fp32 (tcgen05 path)
  int B, N, H, D; float scale;
};
int attn_debug_read(long long* out, int n);
int attn_fwd_launch(const AttnArgs& a, cudaStream_t st);
int attn_bwd_launch(const AttnArgs& a, cudaStream_t st);
// tcgen05 variants (attention_tc.cu): 0 = launched, 1 = shape not covered (D != 64 or N > 256), < 0 = error
int attn_fwd_tc_launch(const AttnArgs& a, cudaStream_t st);
int attn_bwd_tc_launch(const AttnArgs& a, cudaStream_t st);
// rowsum(dO (.) (O + O_lo)) -> a.delta (attention_tc.cu)
int attn_delta_launch(const AttnArgs& a, cudaStream_t st);
// key-tiled tcgen05 variants (attention_long.cu): 0 = launched, 1 = shape not covered (D != 64 or N <= 256), < 0 = error
int attn_fwd_long_launch(const AttnArgs& a, cudaStream_t st);
int attn_bwd_long_launch(const AttnArgs& a, cudaStream_t st);
// key-tiled mma.sync kernels for D = 80 at any N (attention_tiled.cu): 0 = launched, < 0 = error (D != 80 included)
int attn_fwd_tiled_launch(const AttnArgs& a, cudaStream_t st);
int attn_bwd_tiled_launch(const AttnArgs& a, cudaStream_t st);

// fp32.cu: fp32 parity mode (exact-erf GELU forward / backward, attention core forward / backward in SIMT fp32)
int gelu_f32_launch(const float* dy, const float* x, float* out, long n, cudaStream_t st);
int attn_f32_launch(const float* qkv, float* o, float* lse, const float* d_o, float* dqkv, int B, int N, int H, int D,
                    float scale, cudaStream_t st);

// misc.cu
int patchify_launch(const float* img, __nv_bfloat16* out, int B, int Cin, int S, int P, int Kp, cudaStream_t st);
int assemble_launch(const __nv_bfloat16* pe, const float* cls, const float* pos, float* x, int B, int N, int C,
                    cudaStream_t st);
int merge_launch(const float* W, const float* A, const float* Bf, const float* cs, __nv_bfloat16* out, int N, int K,
                 int slices, int R, cudaStream_t st);
int adamw_launch(float* p, const float* g, float* m, float* v, long n, float lr, float b1, float b2, float eps,
                 float wd, int step, float gscale, cudaStream_t st);
int adamw_dev_launch(float* p, const float* g, float* m, float* v, long n, float* state, float b1, float b2, float eps,
                     float wd, float gscale, cudaStream_t st);
int sgemm_launch(const float* A, long ars, long acs, const float* B, long brs, long bcs, float* C, long ldc,
                 const float* bias, int M, int N, int K, float alpha, float beta, float* ws, long ws_floats,
                 cudaStream_t st);

// Per-step staging of the CP factors and its chain rule (misc.cu).  Forward fields first, then the backward's.
struct StageArgs {
  int R, Rp, C, D, L;
  const float *A1, *A3, *A4, *P1, *P2, *R1, *R2, *bias1, *bias2, *bias3;     // CP_* parameters (fp32, contiguous)
  const int *ai, *pi, *mi;                                                   // attn_idx, attn idx, mlp idx per layer
  const float *s_a, *s_m;                                                    // adapter scale per layer
  const float *fb_proj, *fb_fc1, *fb_fc2;                                    // frozen biases stacked over the layers
  float *kr, *cs_qkv, *cs_proj, *cs_fc1, *a_fc2, *cs_fc2, *b_proj, *b_fc1, *b_fc2;   // forward outputs
  float *cs_qkv_pad, *cs_proj_pad, *cs_fc1_pad, *cs_fc2_pad;                 // ... and their [.., Rp] copies (zero padded by the caller)
  const float *g_kr, *g_cs_qkv, *g_cs_proj, *g_cs_fc1, *g_a_fc2, *g_cs_fc2, *g_b_proj, *g_b_fc1, *g_b_fc2;   // incoming gradients (null = none)
  long ld_kr, ld_cs_qkv, ld_cs_proj, ld_cs_fc1, ld_a_fc2, ld_cs_fc2;         // their row pitches (R or Rp)
  float *dA1, *dA3, *dA4, *dP1, *dP2, *dR1, *dR2, *dbias1, *dbias2, *dbias3; // backward outputs (zero filled by the caller)
};
int stage_launch(const StageArgs& a, int backward, cudaStream_t st);

int factor_operands_launch(const float* F, __nv_bfloat16* ext, __nv_bfloat16* t2, long batch, int rows, int R, int Rp,
                           cudaStream_t st);

// GPU input pipeline (preprocess.cu): Pillow-exact bicubic Resize + ToTensor + Normalize on uint8 HWC images
int resize_norm_launch(const uint8_t* src, int B, int H, int W, const int* xbounds, const int* xk, int xksize,
                       const int* ybounds, const int* yk, int yksize, uint8_t* tmp, float* out, uint8_t* out_u8,
                       int OH, int OW, const float* mean, const float* stdv, cudaStream_t st);

}  // namespace cara
