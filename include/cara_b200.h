/* cara_b200 -- C ABI of the B200-native CaRA hot path.
 *
 * The reference (BonnBytes/CaRA) is pure Python: its hot path is the PyTorch code of
 * src/cara/cara.py (cp_attn :15-60, cp_mlp :63-95) and the timm ViT it patches; it has no FFI of its
 * own.  These entry points are what a binding for that path would call instead of the ATen ops listed
 * in SURVEY.md section 2.1: plain pointers and sizes, borrowed device memory (the caller -- PyTorch --
 * owns every buffer; nothing is allocated here), an explicit CUDA stream, int status (0 = ok, <0 =
 * error, text via cara_last_error()).  INTEGRATION.md shows the ctypes binding.
 *
 * All matrices are row-major.  "bf16" = __nv_bfloat16 storage.  Strides (ld*) are in elements.
 */
#ifndef CARA_B200_H_
#define CARA_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define CARA_B200_ABI_VERSION 3
#if defined(__GNUC__)
#define CARA_API __attribute__((visibility("default")))
#else
#define CARA_API
#endif

enum cara_epilogue { CARA_EPI_NONE = 0, CARA_EPI_GELU = 1, CARA_EPI_DGELU = 2, CARA_EPI_DELTA = 3 };

CARA_API int cara_abi_version(void);
CARA_API const char* cara_last_error(void);
/* Select the CUDA device used by subsequent calls from this thread (one process per GPU). */
CARA_API int cara_set_device(int device);

/* Fused CP-adapted projection (replaces cara.py:25-42 qkv, :50-58 proj, :75-82 fc1, :87-93 fc2 and
 * their autograd dX):
 *   out[M,N] = A0[M,K0] * B0[N,K0]^T + bias[N]
 *            + A1[M, slice*K1 : (slice+1)*K1] * B1[N mod (N/ext_slices), K1]^T     (if A1 != NULL)
 * bf16 operands, fp32 accumulation in tensor memory, bf16 outputs.
 *   epi = CARA_EPI_GELU : with u = the bf16-rounded pre-activation: out2 = GELU(u) (exact-erf form, cara.py:84);
 *                         out (NULL for inference) = gelu'(u), kept for backward instead of u
 *   epi = CARA_EPI_DGELU: out = (.) * aux[M,N]          (dX through the fc1 activation: aux = the saved gelu'(u))
 *   epi = CARA_EPI_DELTA: the dX GEMM of the attention OUTPUT projection (out = dO, head dim 64 = one epilogue step)
 *                         also emits the softmax-backward row term the attention backward needs,
 *                         delta[b, h, n] = sum_d bf16(dO)[m, 64h + d] * (aux + aux2)[m, 64h + d],  m = b * seq_n + n,
 *                         with aux / aux2 = the attention output O as its bf16 (hi, lo) pair (cara_attn_fwd's o, o_lo;
 *                         32-byte aligned rows) -- the separate pass over dO and O that cara_attn_bwd otherwise runs
 *                         (autograd of cara.py:47-48) disappears.  N % 64 == 0, M % seq_n == 0.
 * Requirements: K0 % 8 == 0, N % 64 == 0, K1 % 16 == 0, 16-byte aligned bases and row pitches.
 *
 * Side tiles (side != 0): the low-rank operand A1 is itself a contraction of the SAME A0 rows with a [K0, R] factor
 * (cara.py:35,57,81,92: x * delta_W = ((x A) (.) c) B^T), so the kernel computes it too, one extra tile per 128-row
 * panel, from the A0 tiles the panel's output tiles are streaming anyway -- no second pass over x (or g) exists.
 *   side = CARA_SIDE_FWD: T = A0 P^T (P = split(A)^T, bf16 [2*side_rp, K0] = [hi rows ; lo rows]);  side_T (optional,
 *       fp32 [M, side_rp]) = T;  side_U[:, s*3rp : (s+1)*3rp] = split(side_scales[s] (.) T) for s < side_slices.
 *   side = CARA_SIDE_BWD: dU_s = A0[:, s*w : (s+1)*w] P^T per K-slice s (w = K0 / side_slices, P bf16 [2*side_rp, w]);
 *       side_U (bf16 [M, 3rp]) = split(sum_s side_scales[s] (.) dU_s);  side_dc[s] += sum_m dU_s (.) side_T  (fp32,
 *       accumulated;  side_T is an INPUT here: the forward's T).
 * With an adapter segment, side_U must be A1 (the kernel orders the segment's loads after the panel's side tile).
 * N = 0 runs the side tiles alone.  side_rp in {16, 32}; side_slices <= 4; K0 % (64 * K-slices) == 0.
 * sync_ws: CARA_SYNC_WORDS 32-bit words of device memory, zeroed ONCE by the caller and then lent to every call on the
 * same stream (generation counter + four flags per panel; never cleared between calls or graph replays). */
enum cara_side { CARA_SIDE_NONE = 0, CARA_SIDE_FWD = 1, CARA_SIDE_BWD = 2 };
#define CARA_SYNC_WORDS 16386
typedef struct cara_gemm_desc {
  int M, N, K0;
  const void* A0; long lda0;
  const void* B0; long ldb0;
  int K1, ext_slices;
  const void* A1; long lda1;
  const void* B1; long ldb1;
  const float* bias;
  void* out;  int ldo;
  void* out2; int ldo2;
  const void* aux; int ldaux;
  int epi;
  int num_sms; /* 0 = all */
  int side, side_rp, side_slices;
  const void* P; long ldp;
  const float* side_scales;
  float* side_T;
  void* side_U; long side_ldu;
  float* side_dc;
  void* sync_ws;
  const void* aux2; int ldaux2; /* CARA_EPI_DELTA */
  float* delta; int seq_n;      /* CARA_EPI_DELTA: fp32 [M / seq_n, N / 64, seq_n] */
} cara_gemm_desc;
CARA_API int cara_gemm_cp(const cara_gemm_desc* d, void* stream);

/* LayerNorm of timm Block.norm1/norm2/norm (eps 1e-6) fused with the residual stream (replaces the
 * ATen native_layer_norm + add/DropPath kernels of SURVEY 2.1 rows a, m).
 *   x_out = x_in + rowscale[row / rows_per_sample] * delta   (delta NULL: plain LN of x_in)
 *   h = LN(x_out) * gamma + beta;  mean/rstd [M] saved for backward.  x is fp32 [M,C]; delta/h are
 *   bf16 (act_fp32 = 0) or fp32 (act_fp32 = 1).  C must be a multiple of 128. */
CARA_API int cara_ln_fwd(const float* x_in, const void* delta, const float* rowscale, int rows_per_sample,
                         float* x_out, const float* gamma, const float* beta, void* h, float* mean, float* rstd,
                         int M, int C, float eps, int act_fp32, void* stream);
/* dx_out = dx_in + dLN(dh) (gamma/beta frozen);  g_out (optional) = rowscale * dx_out in the activation
 * dtype: the incoming gradient of the branch that fed this residual position. */
CARA_API int cara_ln_bwd(const void* dh, const float* x, const float* mean, const float* rstd, const float* gamma,
                         const float* dx_in, float* dx_out, void* g_out, const float* rowscale, int rows_per_sample,
                         int M, int C, int act_fp32, void* stream);

/* The two LayerNorms above fused with the rank-R row contraction of the projection they feed (bf16 activations):
 * the rows a LayerNorm CTA emits stay in shared memory and are contracted with the (hi, lo) factor there, so the
 * stand-alone pass over the same [M, C] matrix (cara_adapter_rows_fwd / _bwd with K = C resp. N = C, slices = 1) and
 * its launch disappear.  Replaces, besides the LayerNorm, the `x @ A` half of cara.py:35 (qkv, after norm1) and :81
 * (fc1, after norm2), and autograd's `G @ B` for :57 (proj; G = the g_out of norm2's backward) and :92 (fc2; G = the
 * g_out of the next block's norm1 backward).  Operands and outputs exactly as in cara_adapter_rows_fwd / _bwd:
 *   forward : T = h At2^T (fp32 [M,Rp], may be NULL), Uhat[:, s*3Rp:(s+1)*3Rp] = split(scales[s] (.) T), s < slices
 *   backward: dU = g_out Bt2^T, dThat = split(scales[0] (.) dU) (bf16 [M,3Rp]), dscales[0..Rp) += sum_m dU (.) T
 * cara_ln_rows_supported(C, Rp) != 0 for the shapes that keep >= 2 CTAs per SM: (768, 16), (1024, 16). */
CARA_API int cara_ln_rows_supported(int C, int Rp);
CARA_API int cara_ln_fwd_rows(const float* x_in, const void* delta, const float* rowscale, int rows_per_sample,
                              float* x_out, const float* gamma, const float* beta, void* h, float* mean, float* rstd,
                              int M, int C, float eps, const void* At2, const float* scales, int slices, int Rp,
                              float* T, void* Uhat, void* stream);
CARA_API int cara_ln_bwd_rows(const void* dh, const float* x, const float* mean, const float* rstd, const float* gamma,
                              const float* dx_in, float* dx_out, void* g_out, const float* rowscale,
                              int rows_per_sample, int M, int C, const void* Bt2, const float* scales, int Rp,
                              const float* T, void* dThat, float* dscales, void* stream);

/* Rank-R side chain.  Precision convention: factor matrices and low-rank activations are bf16 (hi, lo) pairs
 * (x = hi + lo).  A transposed factor operand "Ft2" is bf16 [2*Rp, K] = [hi rows ; lo rows]; a low-rank
 * activation block is bf16 [.., 3*Rp] = [hi | lo | hi], to be multiplied in cara_gemm_cp (K1 = 3*Rp) against
 * an out-side factor laid out [hi | hi | lo].  Rp = rank zero-padded to 16, 32 or 64.
 *
 * Forward (SURVEY A.1):  T = X A (fp32 [M,Rp]);  Uhat[:, s*3Rp : (s+1)*3Rp] = split(scales[s] (.) T).
 * X bf16 [M,K] (K % 64 == 0); At2 = split(A)^T; scales fp32 [slices,Rp].
 * (cara_gemm_cp can compute the same quantities as side tiles of the projection launch, see there.) */
CARA_API int cara_adapter_rows_fwd(const void* X, long ldx, int M, int K, const void* At2, const float* scales,
                                   int slices, int Rp, float* T, void* Uhat, void* stream);
/* Backward of the same chain (SURVEY A.2): per output slice s, dU_s = G[:, s*w:(s+1)*w] B;
 *   dThat = split(sum_s scales[s] (.) dU_s)  (bf16 [M,3Rp]);  dscales[s] += sum_m dU_s (.) T  (fp32, accumulated).
 * G bf16 [M,N]; Bt2 = split(B)^T bf16 [2Rp, N/slices]. */
CARA_API int cara_adapter_rows_bwd(const void* G, long ldg, int M, int N, int slices, const void* Bt2,
                                   const float* scales, int Rp, const float* T, void* dThat, float* dscales,
                                   void* stream);
/* Factor gradients as skinny contractions over the M tokens (no dW is formed):
 *   out[k mod w, :] += sum_m X[m,k] (Vhi + Vlo)[m, slice k/w]   (w = Kc/slices);  colsum[k] += sum_m X[m,k].
 * X bf16 [M,Kc] (Kc % 256 == 0), V bf16 [M, slices*3Rp] in the [hi | lo | hi] layout; out fp32 [w,Rp] and
 * colsum fp32 [Kc] are accumulated into (caller zeroes them). */
CARA_API int cara_adapter_cols(const void* X, long ldx, int M, int Kc, const void* V, long ldv, int slices, int Rp,
                               float* out, float* colsum, void* stream);

/* Attention core (cara.py:44-48) on the fused projection's [B,N,3,H,D] bf16 output; o is [B,N,H,D].
 * For training also pass lse [B,H,N] fp32 (base-2 log-sum-exp of the scaled scores) and o_lo [B,N,H,D] bf16
 * (the rounding residual of o: o_fp32 = o + o_lo), both consumed by cara_attn_bwd; NULL for inference.
 * D in {64,80}.  D = 64 runs on tcgen05 at every N (N <= 256: one head per CTA pass; N > 256: 128-key tiles);
 * D = 80 runs on mma.sync with the whole head in shared memory: N <= 432, larger N returns an error (cara_attn_tiled_fwd
 * below runs D = 80 at any N). */
CARA_API int cara_attn_fwd(const void* qkv, void* o, void* o_lo, float* lse, int B, int N, int H, int D,
                           float scale, void* stream);
/* delta_ws: caller-provided fp32 workspace [B,H,N] (rowsum(dO (.) O), written by a streaming pre-pass).
 * o == NULL (D = 64 only, any N): delta_ws already holds it -- written by the output projection's dX GEMM
 * (cara_gemm_cp, epi = CARA_EPI_DELTA) -- and the pre-pass is skipped.
 * D = 64 runs on tcgen05 at every N; D = 80 runs on mma.sync with the whole head in shared memory: N <= 320, larger N
 * returns an error (cara_attn_tiled_bwd below runs D = 80 at any N).  Neither uses atomics: dqkv is bit-identical from
 * run to run. */
CARA_API int cara_attn_bwd(const void* qkv, const void* o, const void* o_lo, const float* lse, const void* d_o,
                           void* dqkv, float* delta_ws, int B, int N, int H, int D, float scale, void* stream);
/* The same two calls for D = 80 at any N >= 1 (ViT-H/14 above 224 px), on key-tiled mma.sync kernels: a CTA holds a
 * 128-query (forward), 64-query (dQ) or 64-key (dK/dV) tile and streams the other operand through a two-stage ring of
 * 64-row windows, so shared memory does not grow with N.  Arguments, layouts and outputs are those of cara_attn_fwd /
 * cara_attn_bwd; the backward always runs its own delta pre-pass into delta_ws (o, o_lo and delta_ws are required).
 * Where the whole-head D = 80 calls above also run (forward N <= 432, backward N <= 320), the results are bit-identical
 * to theirs, and a whole-head forward may feed a tiled backward.  No atomics: dqkv is bit-identical from run to run.
 * D != 80, B, N or H <= 0, and a NULL o (or, backward, o_lo / delta_ws) return an error before any launch. */
CARA_API int cara_attn_tiled_fwd(const void* qkv, void* o, void* o_lo, float* lse, int B, int N, int H, int D,
                                 float scale, void* stream);
CARA_API int cara_attn_tiled_bwd(const void* qkv, const void* o, const void* o_lo, const float* lse, const void* d_o,
                                 void* dqkv, float* delta_ws, int B, int N, int H, int D, float scale, void* stream);
/* Profiling aid: copies up to n device-side cycle stamps recorded by the attention kernels (debug builds of the
 * kernels only write them for CTA 0); returns the number of values copied. */
CARA_API int cara_debug_read(long long* out, int n);

/* fp32 mode (north_star: logits rel-err <= 1e-4): plain SIMT fp32, no tensor cores.  Projections run on cara_sgemm,
 * LayerNorm on cara_ln_fwd/bwd with act_fp32 = 1; these two add the exact-erf GELU (cara.py:84) and the attention core
 * (cara.py:44-48) on fp32 [B,N,3,H,D] / [B,N,H,D] tensors (N <= 288, D <= 96; two [N, D+1] fp32 tiles of shared memory).
 *   cara_gelu_f32: dy == NULL -> out = GELU(x);  else out = dy * GELU'(x).
 *   cara_attn_f32: d_o == NULL -> forward (writes o and, if not NULL, lse = natural-log-sum-exp [B,H,N]);
 *                  else backward (reads o, lse, d_o; writes dqkv). */
CARA_API int cara_gelu_f32(const float* dy, const float* x, float* out, long n, void* stream);
CARA_API int cara_attn_f32(const float* qkv, float* o, float* lse, const float* d_o, float* dqkv, int B, int N, int H,
                           int D, float scale, void* stream);

/* Input pipeline of the entry point (reference image_classification/vtab.py:79-82):
 *   transforms.Resize((OH, OW), interpolation=3) -> ToTensor() -> Normalize(mean3, std3)
 * on B decoded uint8 images src [B,H,W,3] (device).  The resize is Pillow's two-pass antialiased bicubic, bit-exact:
 * xbounds/xk (ybounds/yk) are Pillow's integer tap tables for W -> OW (H -> OH): bounds [O,2] = (first tap, taps),
 * k [O, ksize] = 22-bit fixed-point coefficients (cara_b200/preprocess.py builds them; device pointers); pass NULL
 * tables for a dimension that already has the output size.  tmp [B,H,OW,3] uint8 is scratch for the horizontal pass;
 * out [B,3,OH,OW] fp32 and/or out_u8 [B,OH,OW,3] (the resized image before ToTensor) may be NULL.
 * mean3 / std3 are HOST pointers. */
CARA_API int cara_resize_normalize(const unsigned char* src, int B, int H, int W, const int* xbounds, const int* xk,
                                   int xksize, const int* ybounds, const int* yk, int yksize, unsigned char* tmp,
                                   float* out, unsigned char* out_u8, int OH, int OW, const float* mean3,
                                   const float* std3, void* stream);

/* timm PatchEmbed (conv PxP stride P) as im2col: img fp32 [B,Cin,S,S] -> bf16 [B*(S/P)^2, Kp] (zero padded),
 * then cara_gemm_cp against the flattened conv weight, then token assembly with cls/pos into the fp32
 * residual stream x [B,N,C]. */
CARA_API int cara_patchify(const float* img, void* patches, int B, int Cin, int S, int P, int Kp, void* stream);
CARA_API int cara_assemble_tokens(const void* pe, const float* cls, const float* pos, float* x, int B, int N, int C,
                                  void* stream);

/* Staging of one CP factor for the kernels above: F fp32 [batch, rows, R] ->
 *   ext bf16 [batch, rows, 3Rp] = [hi | hi | lo]   (B1 operand of cara_gemm_cp's adapter segment)
 *   t2  bf16 [batch, 2Rp, rows] = [hi^T ; lo^T]    (At2 / Bt2 operand of cara_adapter_rows_*)
 * with hi = bf16(F), lo = bf16(F - hi), zero padded from R to Rp columns. */
CARA_API int cara_factor_operands(const float* F, void* ext, void* t2, long batch, int rows, int R, int Rp,
                                  void* stream);

/* Per-step staging of the twelve CP_* parameters (cara.py:112-125) into the per-layer, per-projection terms of
 * SURVEY A.1 -- what the reference does implicitly when it slices CP_A1 / CP_P1 rows and calls tl.cp_to_tensor
 * (cara.py:26-34, 51-56, 72-80, 88-91) -- and (backward = 1) the chain rule of SURVEY A.2 back to the parameters.
 * One launch each way.  All fp32, contiguous unless a pitch is given; L layers, C = H * D, rank R (Rp = padded).
 *   forward :  kr [C,R] = KR(A3, A4);  cs_qkv [L,3,R] = s_a R1 A1[ai+k];  cs_proj [L,R] = s_a R2 P1[pi];
 *              cs_fc1 [L,4,R] = s_m R2 P1[mi+k];  a_fc2 [L,4C,R] = P1[mi+4+k] (x) P2;  cs_fc2 [L,R] = s_m R2;
 *              b_proj / b_fc1 / b_fc2 = frozen bias + s * CP_bias1/2/3;  *_pad = the cs terms in [.., Rp] rows
 *              (caller zero-fills the padding once).
 *   backward:  g_* (NULL = no gradient; ld_* = row pitch of the R-wide ones) -> dA1, dA3, dA4, dP1, dP2 (the a_fc2
 *              share only), dR1, dR2, dbias1..3, all zero-filled by the caller (indexed rows are added atomically). */
typedef struct cara_stage_desc {
  int R, Rp, C, D, L;
  const float *A1, *A3, *A4, *P1, *P2, *R1, *R2, *bias1, *bias2, *bias3;
  const int *ai, *pi, *mi;
  const float *s_a, *s_m;
  const float *fb_proj, *fb_fc1, *fb_fc2;
  float *kr, *cs_qkv, *cs_proj, *cs_fc1, *a_fc2, *cs_fc2, *b_proj, *b_fc1, *b_fc2;
  float *cs_qkv_pad, *cs_proj_pad, *cs_fc1_pad, *cs_fc2_pad;
  const float *g_kr, *g_cs_qkv, *g_cs_proj, *g_cs_fc1, *g_a_fc2, *g_cs_fc2, *g_b_proj, *g_b_fc1, *g_b_fc2;
  long ld_kr, ld_cs_qkv, ld_cs_proj, ld_cs_fc1, ld_a_fc2, ld_cs_fc2;
  float *dA1, *dA3, *dA4, *dP1, *dP2, *dR1, *dR2, *dbias1, *dbias2, *dbias3;
} cara_stage_desc;
CARA_API int cara_stage_terms(const cara_stage_desc* d, int backward, void* stream);

/* Eval-mode merge (SURVEY A.3; the reference re-materialises the delta every forward, cara.py:27,52,76,88):
 *   Weff[n,k] = W[n,k] + sum_r Bf[n mod w, r] cs[n / w, r] A[k, r],  W fp32 [N,K] -> Weff bf16 [N,K]. */
CARA_API int cara_merge_weights(const float* W, const float* A, const float* Bf, const float* cs, void* Weff, int N,
                                int K, int slices, int R, void* stream);

/* torch.optim.AdamW update (vit_cp.py:185) over one flat fp32 buffer; grads are pre-multiplied by gscale. */
CARA_API int cara_adamw_step(float* p, const float* g, float* m, float* v, long n, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int step, float gscale, void* stream);

/* The same update with its two per-step scalars in DEVICE memory, so that the launch can be part of a replayed CUDA
 * graph (the whole vit_cp.py:45-50 iteration -- zero_grad, forward, CE, backward, gradient all-reduce, AdamW -- is then
 * one graph launch): state is fp32[4] = { learning rate, optimizer steps taken so far, exit ticket (zero), unused }.
 * The kernel uses step = state[1] + 1 for the bias corrections and stores it back; the host rewrites state[0]
 * (stream-ordered) whenever the schedule changes the rate (vit_cp.py:55-56). */
CARA_API int cara_adamw_step_dev(float* p, const float* g, float* m, float* v, long n, float* state, float beta1,
                                 float beta2, float eps, float weight_decay, float gscale, void* stream);

/* Plain fp32 GEMM with general strides for the tiny trainable head (vit_cp.py:166):
 *   C[m,n] = alpha * sum_k A[m*ars + k*acs] * B[k*brs + n*bcs] + beta * C[m,n] + bias[n].
 * workspace (optional, device, workspace_floats fp32 elements, borrowed for the call): lets small problems split K
 * over more CTAs; the partial sums are reduced in a fixed order, so results are reproducible bit for bit. */
CARA_API int cara_sgemm(const float* A, long ars, long acs, const float* B, long brs, long bcs, float* C, long ldc,
                        const float* bias, int M, int N, int K, float alpha, float beta, float* workspace,
                        long workspace_floats, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CARA_B200_H_ */
