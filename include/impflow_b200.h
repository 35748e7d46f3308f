/*
 * impflow_b200.h — C ABI of libimpflow_b200.so (sm_100a).
 *
 * The reference (musikisomorphie/implicit-normalizing-flows) has no FFI: its boundary for the
 * hot path is the Python module API (SURVEY.md §8b).  This header is the C-ABI layer the
 * Python host classes in `implicit-normalizing-flows_b200/` bind with ctypes; every entry
 * point names the reference code it replaces (file:line relative to the reference root).
 *
 * Conventions
 *  - all tensor arguments are DEVICE pointers to dense fp32 unless stated; the caller
 *    (PyTorch) owns every buffer including workspaces; nothing here allocates or frees.
 *  - `stream` is a cudaStream_t passed as void*; launches are asynchronous on it and never
 *    synchronise unless stated.
 *  - return 0 on success, negative on error; the message is available through
 *    impflow_last_error() (thread-local).
 */
#ifndef IMPFLOW_B200_H
#define IMPFLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IMPFLOW_ABI_VERSION 1

/* activation kinds (lib/layers/base/activations.py:7-12 Sin, :64-71 Swish; torch.nn.ReLU) */
#define IMPFLOW_ACT_NONE 0
#define IMPFLOW_ACT_SIN 1
#define IMPFLOW_ACT_LIPSWISH 2
#define IMPFLOW_ACT_RELU 3
/* pseudo kind for the dmul_pre epilogues: dmul_pre already holds the multiplier act'(pre) (evaluated once per
 * saved forward by impflow_act_mul order 1), so the epilogue is one multiply instead of an exp + divide */
#define IMPFLOW_ACT_MULTIPLIER 4

int impflow_version(void);
const char* impflow_last_error(void);
/* number of kernels launched by this library in this process so far (bench.py gpu_launches) */
long long impflow_launch_count(void);
/* kernels of this library launched by replaying a CUDA graph the host captured (they do not pass the launchers) */
void impflow_add_launch_count(long long n);

/* ------------------------------------------------------------------------------------------
 * Broyden solver algebra — replaces lib/layers/broyden.py:101-193 (rmatvec, matvec, the
 * rank-1 update, norms, best-iterate tracking, break rules).  g itself is evaluated by the
 * caller between calls.  History is kept as U^T (B,T,d) and V^T (B,T,d), row-contiguous.
 *
 * Device state (int32/float/double words, see BroydenState in csrc/broyden.cu):
 *   the caller allocates impflow_broyden_state_bytes(T) bytes and may copy it to the host to
 *   read nstep / lowest_step / flags / trace.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t nstep;        /* iterations done (broyden.py:155) */
  int32_t lowest_step;  /* step of the best iterate (:162) */
  int32_t active;       /* 1 while the while-condition (:153) still holds */
  int32_t prot_break;   /* protective break fired (:169-172) */
  int32_t converged;    /* objective < eps (:163) */
  int32_t stagnated;    /* stagnation rule fired (:165-168) */
  int32_t do_update;    /* the last step must apply the rank-1 update (:174-181) */
  int32_t new_lowest;   /* the last step improved the best iterate (:159-162) */
  int32_t threshold;
  int32_t counter;      /* internal: last-block election */
  double eps;           /* eps * sqrt(B*d) (:131) */
  double init_objective;
  double lowest;
  double objective;     /* latest ||g||_F */
  double trace[64];     /* trace[0..nstep]; threshold <= 63 */
} impflow_broyden_state;

size_t impflow_broyden_state_bytes(void);

/* After the caller evaluated g0 = g(x0):  init state, low_x=x0, low_g=g0, xn = x0 + (-g0)
 * (broyden.py:136-151).  sample_sq (B) receives per-sample ||g0||^2, low_sq (B) a copy;
 * `partial` is a float workspace of impflow_broyden_workspace_floats(B,d,T) elements. */
int impflow_broyden_begin(const float* x0, const float* g0, float* xn, float* low_x, float* low_g,
                          float* sample_sq, float* low_sq, float* partial, impflow_broyden_state* state,
                          int B, long long d, int threshold, double eps_scaled, void* stream);

/* After the caller evaluated gn = g(xn): one loop body of broyden.py:153-181.
 *  - norms + bookkeeping + break rules on the device (state updated);
 *  - if the step must update: v^T, u (NaN scrub), store in slot (nstep-1), next direction,
 *    and x_next = xn + update is written into `x_old`'s buffer (the caller then swaps roles:
 *    x_old<->xn, g_old<->gn);
 *  - if the step improved the best iterate: low_x=xn, low_g=gn, low_sq=sample_sq.
 * `partial` is a float workspace of impflow_broyden_workspace_floats(B,d,T) elements. */
size_t impflow_broyden_workspace_floats(int B, long long d, int threshold);
int impflow_broyden_step(float* x_old, const float* g_old, const float* xn, const float* gn, float* Ut,
                         float* Vt, float* low_x, float* low_g, float* sample_sq, float* low_sq,
                         float* partial, impflow_broyden_state* state, int B, long long d, int threshold,
                         void* stream);

/* Persistent small-d solver (toy / tabular MLP branches, d <= 128, widths <= 256): ONE cooperative
 * launch runs the whole solve of x_embed - f(z) - z = 0 — branch evaluations (fused fp32 MLP with the
 * activation `act_kind` between its L linear layers), batch-global norms, break rules, best iterate and
 * rank-1 updates — replacing the host-driven loop of broyden.py:123-193 + implicit_block.py:68-80.
 *   Wt[l]  : DEVICE pointer to the transposed effective weight [dims[l]][dims[l+1]] (HOST array of L)
 *   bias[l]: DEVICE pointer or NULL (HOST array of L, or NULL)
 *   beta_sp[l]: DEVICE scalar softplus(beta) of the LipSwish module behind layer l, l < L-1 (HOST array of L-1
 *            pointers; every Swish owns its own learnable beta, activations.py:64-71); NULL for Sin / ReLU
 *   za     : start point z0 (B,d) on entry; za/ga/zb/gb are (B,d) scratch afterwards
 *   low_z  : best iterate on return; state: as in impflow_broyden_step
 *   partial: impflow_mlp_solver_partial_doubles() doubles of workspace */
int impflow_mlp_solver_limits(int* max_layers, int* max_width, int* max_d);
size_t impflow_mlp_solver_partial_doubles(void);
int impflow_mlp_broyden_solve(const float* x_embed, const float* const* Wt, const float* const* bias,
                              const int* dims, int L, int act_kind, const float* const* beta_sp, float* za, float* ga,
                              float* zb, float* gb, float* low_z, float* low_g, float* Ut, float* Vt,
                              float* sample_sq, float* low_sq, double* partial, impflow_broyden_state* state,
                              int B, int threshold, double eps_scaled, void* stream);

/* Implicit-backward solve v^T (I + J_f(z)) = rhs of the same MLP branch (imBlock.Backward,
 * implicit_block.py:199-207) in the same persistent kernel: the residual is g(v) = v^T J + v - rhs with
 * v^T J = (((v W_{L-1}) * D_{L-1}) W_{L-2} * D_{L-2}) ... W_0, D_l = act'(pre-activation in front of layer l).
 *   W[l]   : DEVICE pointer to the effective weight of layer l, [dims[l+1]][ldw[l]] row-major (HOST array of L)
 *   dmul[l]: DEVICE pointer to D_l, (B, dims[l]) contiguous, or NULL (HOST array of L; dmul[0] must be NULL)
 *   za     : start point (zeros in the reference) on entry; other buffers / state as in impflow_mlp_broyden_solve */
int impflow_mlp_broyden_solve_vjp(const float* rhs, const float* const* W, const int* ldw, const float* const* dmul,
                                  const int* dims, int L, float* za, float* ga, float* zb, float* gb, float* low_z,
                                  float* low_g, float* Ut, float* Vt, float* sample_sq, float* low_sq, double* partial,
                                  impflow_broyden_state* state, int B, int threshold, double eps_scaled, void* stream);

/* One-launch power series of a small-d MLP branch at a saved point and for one probe v — the training path of the
 * basic estimator (implicit_block.py:418-426 with create_graph=True, taken graph-free):
 *     Ls (n+1, B, d): l_0 = v, l_k = (J^T)^k v      Rs (n, B, d): r_0 = v, r_m = J^m v
 *     S (B) = sum_k c_k <l_k, v>                    Wm (n, B, d): w_m = sum_{a=0}^{n-1-m} c_{a+m} l_a
 *   W[l], ldw[l]: effective weight of layer l, [dims[l+1]][ldw[l]] row-major;  Wt[l]: its transpose
 *   [dims[l]][dims[l+1]] contiguous;  dmul[l]: act'(pre-activation in front of layer l), (B, dims[l]), dmul[0] NULL
 *   (HOST arrays of L DEVICE pointers);  coeffs: n HOST doubles, n <= 32.  Same limits as the persistent solver. */
int impflow_mlp_series(const float* v, const float* const* W, const int* ldw, const float* const* Wt,
                       const float* const* dmul, const int* dims, int L, int B, int n, const double* coeffs,
                       float* Ls, float* Rs, float* Wm, float* S, void* stream);

/* ------------------------------------------------------------------------------------------
 * Elementwise / reductions on the path
 * ------------------------------------------------------------------------------------------ */
/* out = g * act^(order)(x) (g may be NULL -> 1).  order 0..3; beta_sp = DEVICE pointer to the
 * scalar softplus(beta) for LipSwish (NULL otherwise) — a pointer so that no host sync is needed.  Replaces activations.py:11-12,70-71 and their autograd derivatives. */
int impflow_act_mul(const float* x, const float* g, float* out, long long n, int kind, int order,
                    const float* beta_sp, void* stream);
/* hi + lo = act^(order)(x) as tf32 planes (the K-major / MN-major operand form of the tensor-core kernels). */
int impflow_act_split(const float* x, float* hi, float* lo, long long n, int kind, int order, const float* beta_sp,
                      void* stream);
/* out[0] = sum_i g[i] * g2[i] * d/d(beta_sp) act^(order)(x[i])  (order 0..2; g2 may be NULL);
 * deterministic 2-stage reduce; `partial` needs impflow_reduce_workspace_floats(n) floats. */
size_t impflow_reduce_workspace_floats(long long n);
int impflow_act_beta_grad(const float* x, const float* g, const float* g2, float* out, float* partial,
                          long long n, int order, const float* beta_sp, void* stream);
/* out = act''(p) * t * ga + act'(p) * gb (gb may be NULL): the activation step of the hand-derived
 * reverse pass of the Neumann gradient estimator (implicit_block.py:386-388, 429-438). */
int impflow_act_second(const float* p, const float* t, const float* ga, const float* gb, float* out,
                       long long n, int kind, const float* beta_sp, void* stream);
/* The activation step of that reverse sweep for one LipSwish layer in ONE pass over (M,N) tensors:
 *   ybar = act''(p) t ta + act'(p) ab   written as tf32 hi/lo planes (they feed the next transposed GEMM and the
 *   weight gradient), colsum[n] = sum_m ybar (bias gradient of the layer below), beta_grad[0] = sum ta t
 *   d/dbeta act'(p) + ab d/dbeta act(p).  ab may be NULL.  ws: impflow_neumann_act_bwd_workspace_floats(M,N). */
size_t impflow_neumann_act_bwd_workspace_floats(long long M, int N);
int impflow_neumann_act_bwd(const float* p, const float* t, const float* ta, const float* ab, float* y_hi, float* y_lo,
                            float* colsum, float* beta_grad, float* ws, long long M, int N, const float* beta_sp,
                            void* stream);
/* out = a*ca + b*cb + c*cc (b, c may be NULL). Solver residuals x_embed - f(z) - z
 * (implicit_block.py:72) and v J + v - grad (:199-203); Neumann accumulation (:435). */
int impflow_lincomb3(const float* a, float ca, const float* b, float cb, const float* c, float cc,
                     float* out, long long n, void* stream);
/* out[b] = beta*out[b] + alpha * <a[b,:], c[b,:]>  — Hutchinson trace term
 * (implicit_block.py:423,437). */
int impflow_rowdot(const float* a, const float* c, float* out, int B, long long d, float alpha, float beta,
                   void* stream);
/* out[n] = sum_m a[m,n]  (bias gradient); two deterministic stages over row chunks, `partial`
 * holds impflow_colsum_chunks(M,N) * N floats (may be NULL when that is 1). */
int impflow_colsum_chunks(long long M, int N);
int impflow_colsum(const float* a, float* out, float* partial, long long M, int N, void* stream);
/* out[n,m] = a[m,n] */
int impflow_transpose(const float* a, float* out, long long M, long long N, void* stream);
/* NHWC 3x3, stride 1, pad 1 patch gather col[(b,y,x),(ky,kx,c)] = x[b,y+ky-1,x+kx-1,c] (rows of
 * `ld` >= 9*C floats, the tail zero-filled so that K can be padded to a multiple of 32), and its
 * adjoint (scatter-sum) with the same fused epilogue as impflow_gemm_nt (N = C, ldc = C). */
int impflow_im2col3x3(const float* x, float* col, int B, int H, int W, int C, int ld, void* stream);
/* the same gather written directly as tf32 hi/lo planes (the A operand of impflow_gemm_nt_tc) */
int impflow_im2col3x3_split(const float* x, float* col_hi, float* col_lo, int B, int H, int W, int C, int ld,
                            void* stream);
int impflow_col2im3x3(const float* col, int B, int H, int W, int C, const float* bias, float* pre_out,
                      float* act_out, const float* dmul_pre, int act_kind, const float* beta_sp, void* stream);

/* Step tail over FLAT parameter / gradient / moment buffers in one pass — replaces clip_grad_norm_
 * (train_img.py:652), the vendored Adam update (lib/optimizers.py:47-107: denom = sqrt(v) + eps) and the EMA
 * of the parameters (lib/utils.py:140-146, train_img.py:658).  gnorm_sq: DEVICE scalar sum(g^2) (e.g. from
 * impflow_rowdot), NULL or max_norm <= 0 = no clipping; g is overwritten with the clipped gradient; ema may
 * be NULL; step_size = lr * sqrt(1 - beta2^t) / (1 - beta1^t) is computed by the host. */
int impflow_clip_adam_ema(float* p, float* g, float* m, float* v, float* ema, long long n, const float* gnorm_sq,
                          float max_norm, float step_size, float beta1, float beta2, float eps, float ema_decay,
                          void* stream);

/* ActNorm1d / ActNorm2d (lib/layers/act_norm.py:39-62), the layer in front of every imBlock
 * (implicit_flow.py:411-428; SURVEY.md section 8(f) row 1).  x, y, gy, gx: (B, C, HW) contiguous (HW = 1 for the 1d
 * case) or, with channels_last = 1, (B, HW, C) — the order the branch kernels leave their outputs in.
 *   forward : y = (x + bias_c) * exp(weight_c);  logpx_out[b] = logpx[b] - HW * sum_c weight_c  (both NULL: y only)
 *   backward: gx = gy * exp(weight_c);  gbias_c = sum gy * exp(weight_c);
 *             gweight_c = sum gy * y - HW * sum_b g_logpx[b]   (g_logpx may be NULL); fixed-order reductions.
 * ws: impflow_actnorm_workspace_floats(C) floats. */
int impflow_actnorm_forward(const float* x, const float* bias, const float* weight, float* y, const float* logpx,
                            float* logpx_out, long long B, int C, long long HW, int channels_last, void* stream);
size_t impflow_actnorm_workspace_floats(int C);
int impflow_actnorm_backward(const float* gy, const float* y, const float* weight, const float* g_logpx, float* gx,
                             float* gbias, float* gweight, float* ws, long long B, int C, long long HW,
                             int channels_last, void* stream);

/* ------------------------------------------------------------------------------------------
 * Residual-branch contractions — replace F.linear / F.conv2d and their vjps
 * (mixed_lipschitz.py:134-136, 388-391; implicit_block.py:422,434,436).
 *   C[M,N] = A[M,K] * B[N,K]^T  (+ bias[N])   fp32 in / fp32 accumulate.
 * Epilogue (all optional, NULL = off):
 *   pre_out  <- acc + bias                       (pre-activation, kept for the vjp)
 *   act_out  <- act(acc + bias)                  (input of the next layer)
 *   dmul_pre : if set, pre_out <- acc * act'(dmul_pre[m,n])   (vjp / tangent through the activation)
 *              and act_out (if given) <- acc, the raw product
 * impflow_gemm_nt     : exact-fp32 CUDA-core tiles (any M,N,K; small MLP shapes, cross-check).
 * impflow_gemm_nt_tc  : tcgen05 3xTF32 (TMA-fed, TMEM accumulators).  Operands come as tf32 hi/lo
 *                       planes (a = hi + lo, see impflow_split_tf32); needs K % 32 == 0 and rows that
 *                       are 16-byte aligned (returns -2 otherwise).  split_hi/split_lo (optional)
 *                       receive the hi/lo planes of the value that feeds the next GEMM
 *                       (act_out value, or the act' product in dmul mode).
 * ------------------------------------------------------------------------------------------ */
int impflow_gemm_nt(const float* A, long long lda, const float* Bm, long long ldb, const float* bias,
                    float* pre_out, float* act_out, const float* dmul_pre, long long ldc, long long M,
                    int N, int K, int act_kind, const float* beta_sp, void* stream);
/* Exact-fp32 CUDA-core GEMM with element strides, C[m,n] = sum_k A[m*sAm + k*sAk] * B[n*sBn + k*sBk] (+ bias[n]):
 * the autograd primitives of the small shapes use it for A B, A^T B, A B^T, A^T B^T without transposed copies. */
int impflow_gemm_strided(const float* A, long long sAm, long long sAk, const float* Bm, long long sBn, long long sBk,
                         const float* bias, float* out, long long ldc, long long M, int N, int K, void* stream);
/* Exact-fp32 weight-gradient contraction dW[N1,N2] = G[M,N1]^T A[M,N2] straight from the row-major operands, split
 * along the M rows over the SMs with a fixed-order reduce (small / ragged shapes: the MLP flows' 128-wide layers over
 * n x batch rows, where impflow_wgrad_tc does not apply).  ws: impflow_wgrad_simt_workspace_floats(M, N1, N2) floats. */
size_t impflow_wgrad_simt_workspace_floats(long long M, int N1, int N2);
int impflow_wgrad_simt(const float* G, long long ldg, const float* A, long long lda, float* out, long long ldo,
                       long long M, int N1, int N2, float* ws, void* stream);
int impflow_gemm_nt_tc(const float* A_hi, const float* A_lo, long long lda, const float* B_hi,
                       const float* B_lo, long long ldb, const float* bias, float* pre_out, float* act_out,
                       const float* dmul_pre, float* split_hi, float* split_lo, long long ldc, long long M,
                       int N, int K, int act_kind, const float* beta_sp, float* splitk_ws, void* stream);
/* Weight-gradient shapes (small M x N, K = all pixels) are split along K over the SMs: with the plain
 * epilogue (pre_out (+bias) only) and a workspace of impflow_gemm_tc_splits(M,N,K) * M * N floats the
 * kernel writes per-slice partials and a fixed-order reduce finishes; splitk_ws = NULL disables it. */
int impflow_gemm_tc_splits(long long M, int N, int K);
/* Epilogue switch for A/B measurements: 1 (default) = outputs staged in shared memory and written by bulk tensor
 * (TMA) stores, 0 = per-thread 32-byte global stores.  Returns the previous setting. */
int impflow_gemm_tc_set_tma_store(int on);
/* CTA-pair switch for A/B measurements: 1 (default) = problems with N >= 256 that fill the 74 TPCs run on
 * clusters of two CTAs (tcgen05.mma.cta_group::2, 256x256 tiles, each CTA stages half of the weight tile),
 * 0 = single-CTA tiles only.  Returns the previous setting. */
int impflow_gemm_tc_set_pair(int on);
/* Programmatic dependent launch of the tile kernels (k_gemm_tc3, k_branch3): 1 (default) = they are launched with
 * the stream-serialisation attribute, so their set-up (barriers, tensor memory, tensor-map prefetch) overlaps the
 * tail of the preceding kernel and every thread executes griddepcontrol.wait before the first global-memory access;
 * 0 = ordinary launches.  Returns the previous setting. */
int impflow_set_pdl(int on);
/* Weight-gradient contraction dW[N1,N2] = G[Mpix,N1]^T A[Mpix,N2] (K = all pixels) straight from the row-major
 * hi/lo planes: both operands are fed to tcgen05 as MN-major tiles (TMA boxes of 32 pixels x 32 channels), so
 * no transposed copies are made (replaces the autograd weight gradients of F.conv2d / F.linear,
 * mixed_lipschitz.py:134-136,388-391).  Needs Mpix % 32 == 0 and 16-byte aligned rows (-2 otherwise);
 * out[n1*ldo + n2] (or out[n2*ldo + n1] when transpose_out) receives the fixed-order sum of the split-K
 * partials; ws holds impflow_wgrad_tc_workspace_floats() floats. */
size_t impflow_wgrad_tc_workspace_floats(long long Mpix, int N1, int N2);
/* A/B switch: 1 (default) = work items in slice-major order (all output tiles of a K slice side by side: every
 * operand slice leaves DRAM once), 0 = tile-major (round 1).  Returns the previous setting. */
int impflow_wgrad_set_slice_major(int on);
int impflow_wgrad_tc(const float* G_hi, const float* G_lo, long long ldg, const float* A_hi, const float* A_lo,
                     long long lda, float* out, long long ldo, int transpose_out, long long Mpix, int N1, int N2,
                     float* ws, void* stream);
/* a -> tf32 "hi" (round-to-nearest) and "lo" = a - hi planes used by the 3xTF32 backend. */
int impflow_split_tf32(const float* a, float* hi, float* lo, long long n, void* stream);
/* out_hi/out_lo[n,m] = tf32 split of a[m,n] (a is M x N row-major): the K-major operand planes of the
 * weight-gradient GEMMs dW = G^T A (K = all pixels) in one pass. */
int impflow_transpose_split(const float* a, float* out_hi, float* out_lo, long long M, long long N, void* stream);

/* Fused residual-branch tile kernel for the 3x3 / 1x1 / 3x3 conv branch whose narrow side has 9*c <= 32
 * tap columns (implicit_flow.py:359-398 at the first CIFAR scale), forward or transposed (vjp), one launch:
 *     Y[M,N3] (+)= psi2( psi1( X0[M,32] W1[C,32]^T ) W2[C,C]^T ) W3[N3,C]^T
 *   psi_l(t) = act(t + bias_l)  with pre_l_out <- t + bias_l (optional)     when mul_l == NULL   (forward)
 *   psi_l(t) = t * mul_l[m,n]   (mul_l = act'(pre), evaluated once per saved forward)             (vjp)
 * The C-wide intermediates stay in tensor memory; weights come as tf32 hi/lo planes (K-major rows);
 * X0 is plain fp32 (im2col of the narrow tensor, ldx >= 32, columns >= 9c zero).  Needs C % 256 == 0 and
 * N3 <= 32 (returns -2 otherwise).  When C > 256 the two 256-channel halves are summed into `out` with
 * atomics: the caller zero-fills `out` (two addends on zero: order-independent, deterministic).
 * Replaces three impflow_gemm_nt_tc launches + the plane traffic between them. */
int impflow_branch3_tc(const float* x0, long long ldx, const float* W1_hi, const float* W1_lo, const float* W2_hi,
                       const float* W2_lo, const float* W3_hi, const float* W3_lo, const float* bias1,
                       const float* bias2, const float* mul1, const float* mul2, float* pre1_out, float* pre2_out,
                       float* out, long long ldo, long long M, int C, int N3, int act_kind, const float* beta1,
                       const float* beta2, void* stream);

/* Fused layers 2 + 3 of the same branch for the wider scales (9c = 108 / 432 tap columns; implicit_flow.py:359-398
 * at c = 12 / 48), forward or transposed, one launch (csrc/chain23_fused.cu):
 *     out_q[M,N3] = psi2( A1[M,C] W2[C,C]^T )[:, q] W3[N3, q]^T      for every 128-channel quarter q of layer 2
 *   A1 comes as the tf32 hi/lo planes the layer-1 GEMM (impflow_gemm_nt_tc, split outputs) wrote; psi2 as in
 *   impflow_branch3_tc (bias2 + activation with optional pre2_out, or * mul2).  The C-wide layer-2 output stays in
 *   tensor memory.  `out` receives impflow_chain23_parts(C) = C/128 PARTIAL results, part_stride floats apart
 *   (>= M*ldo); the caller sums them in fixed order (impflow_conv3_* do it in the col2im epilogue).
 * Needs C % 128 == 0 and 16-byte aligned rows (returns -2 otherwise).  Replaces two impflow_gemm_nt_tc launches and
 * the plane traffic between them. */
int impflow_chain23_parts(int C);
/* A_lo = NULL: A_hi is the plain fp32 layer-2 input; the kernel splits every landed chunk into hi / lo on chip. */
int impflow_chain23_tc(const float* A_hi, const float* A_lo, long long lda, const float* W2_hi, const float* W2_lo,
                       const float* W3_hi, const float* W3_lo, const float* bias2, const float* mul2, float* pre2_out,
                       float* out, long long ldo, long long part_stride, long long M, int C, int N3, int act_kind,
                       const float* beta2, void* stream);

/* ------------------------------------------------------------------------------------------
 * Native host runtime of the 3x3 / 1x1 / 3x3 conv residual branch (implicit_flow.py:359-398): one C call per
 * branch evaluation, per Neumann power-series chain and per Broyden solve (csrc/conv3_plan.cu).  All
 * tensors are NHWC "rows": M = B*H*W rows of c floats; a sample is a contiguous block of H*W*c floats.
 * Shapes with 9c <= 32 and C % 256 == 0 run on impflow_branch3_tc, the others on im2col planes + the layer-1
 * impflow_gemm_nt_tc + impflow_chain23_tc (C % 128 == 0; else two more GEMMs) + col2im.  The caller owns every buffer; `ws` holds
 * impflow_conv3_workspace_floats(B,H,W,c,C,k0) floats and may be shared by all plans used on one stream.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t B, H, W;       /* images and their spatial size */
  int32_t c, C;          /* narrow (input = output) channels, hidden width */
  int32_t k0;            /* 9c rounded up to a multiple of 32: row length of the patch matrices */
  int32_t act_kind;      /* activation between the layers (one kind for both) */
  int32_t act0_kind;     /* leading activation, IMPFLOW_ACT_NONE if the branch starts with the conv */
  int32_t allow_fused;   /* 0 = never use the one-launch tile kernel (A/B switch) */
  int32_t reserved;
  const float *beta0, *beta1, *beta2; /* device scalars softplus(beta) of the three LipSwish modules or NULL */
  const float *W1f_hi, *W1f_lo;       /* (C, k0)  layer 1, rows (ky,kx,ci) zero-padded to k0 */
  const float *W2f_hi, *W2f_lo;       /* (C, C)   layer 2 */
  const float *W3f_hi, *W3f_lo;       /* (9c, C)  layer 3 in tap-major GEMM form (col2im follows) */
  const float *b1, *b2, *b3;          /* biases (C), (C), (c) or NULL */
  const float *W3b_hi, *W3b_lo;       /* (C, k0)  transposed layer 3 */
  const float *W2b_hi, *W2b_lo;       /* (C, C)   transposed layer 2 */
  const float *W1b_hi, *W1b_lo;       /* (9c, C)  transposed layer 1 */
  float* ws;
} impflow_conv3_plan;

size_t impflow_conv3_workspace_floats(int B, int H, int W, int c, int C, int k0);
/* y_rows = nnet(x_rows); pre1 / pre2 (M,C; optional) receive the hidden pre-activations kept for the vjp */
int impflow_conv3_forward(const impflow_conv3_plan* plan, const float* x_rows, float* y_rows, float* pre1,
                          float* pre2, void* stream);
/* d_l = act'(pre_l): the multipliers of the transposed sweep, evaluated once per saved forward */
int impflow_conv3_prepare_vjp(const impflow_conv3_plan* plan, const float* pre1, const float* pre2, float* d1,
                              float* d2, void* stream);
/* out_rows = v^T J at the saved point; pre0 = the branch input rows (needed when act0_kind != NONE) */
int impflow_conv3_vjp(const impflow_conv3_plan* plan, const float* pre0, const float* d1, const float* d2,
                      const float* v_rows, float* out_rows, void* stream);
/* The n-term vjp chain v^T J^k of the power-series estimators in ONE call, with both accumulations fused into
 * the chain (no separate linear-combination launches):
 *   w_rows  (optional, with coeffs):     w = v + sum_k coeffs[k-1] * v^T J^k     — the no-grad Neumann sum of the
 *                                         gradient estimator (implicit_block.py:431-435), added in the col2im epilogue
 *   dot_out (optional, with dot_coeffs): dot_out[b] = sum_k dot_coeffs[k-1] * <v^T J^k, v>_b — the Hutchinson terms
 *                                         of the basic estimator (:418-426, eval mode)
 * coeffs / dot_coeffs are HOST arrays of n doubles; at least one of the two outputs must be requested. */
int impflow_conv3_power_series(const impflow_conv3_plan* plan, const float* pre0, const float* d1, const float* d2,
                               const float* v_rows, const double* coeffs, int n, float* w_rows,
                               const double* dot_coeffs, float* dot_out, void* stream);
/* Whole Broyden solve (broyden.py:123-193) with the residual evaluated by this branch:
 *   mode 0: g(z) = rhs - nnet(z) - z        (forward / inverse solve, implicit_block.py:68-80; rhs = x_embed)
 *   mode 1: g(v) = v^T J + v - rhs          (implicit backward, :199-207; rhs = incoming gradient)
 * xa holds the start point; xa/xb/ga/gb are (B,d) scratch; the other buffers are those of
 * impflow_broyden_step.  The loop is SYNC-FREE: the residual (branch evaluation + the x_embed - f - z / vJ + v - grad
 * combination in the col2im epilogue), the norms, the reference's break rules (broyden.py:153-181) and the rank-1
 * update all run on the device; the host enqueues up to `runahead` iterations (impflow_conv3_set_runahead, default 2)
 * beyond the last decision it has seen, kernels enqueued behind the end of the loop turn into no-ops through a
 * device-side gate, and the host learns each decision from a progress record the decision kernel writes into mapped
 * pinned host memory.  The stream is drained ONCE per solve, for the final state record.
 * state_host: PINNED host memory of impflow_conv3_broyden_host_bytes(threshold) bytes (state record + progress
 * records); on return it starts with the final state and low_x holds the best iterate. */
size_t impflow_conv3_broyden_host_bytes(int threshold);
/* A/B switch: 1 (default) = layers 2 + 3 of the wider scales run as impflow_chain23_tc, 0 = two GEMM launches.
 * Returns the previous setting. */
int impflow_conv3_set_chain23(int on);
/* A/B switch: 1 = the layer-1 GEMM in front of impflow_chain23_tc writes ONE fp32 plane and the fused kernel
 * derives the tf32 hi / lo planes in shared memory (A_lo = NULL), 0 (default: measured faster, the fused kernel is
 * bound by the shared-memory port) = hi / lo planes through HBM.  Same roundings, bit-identical results.  Returns the
 * previous setting. */
int impflow_conv3_set_chain23_a32(int on);
/* A/B switch: iterations enqueued ahead of the device's decision (0 = copy the state and synchronise the stream after
 * every iteration, the round-1 behaviour).  Returns the previous setting. */
int impflow_conv3_set_runahead(int iterations);
/* A/B switch: 1 (default) = in impflow_conv3_power_series the col2im epilogue of term k also writes the im2col rows
 * (and clears the tap accumulator) of term k + 1, so every term but the first is two launches (tile kernel) instead
 * of three; 0 = a k_conv3_in launch per term.  Same values either way.  Returns the previous setting. */
int impflow_conv3_set_chain_fuse(int on);
int impflow_conv3_broyden(const impflow_conv3_plan* plan, int mode, const float* rhs_rows, const float* pre0,
                          const float* d1, const float* d2, float* xa, float* xb, float* ga, float* gb, float* low_x,
                          float* low_g, float* Ut, float* Vt, float* sample_sq, float* low_sq, float* partial,
                          impflow_broyden_state* state_dev, impflow_broyden_state* state_host, int threshold,
                          double eps_scaled, void* stream);

/* ------------------------------------------------------------------------------------------
 * Induced 2-norm power iteration for a dense (out,in) matrix — replaces
 * mixed_lipschitz.py:85-123 (Linear) and :276-319 (1x1 conv).  One CTA, device-side early
 * exit with the reference tolerance rule; u, v updated in place; sigma[0] = u^T W v,
 * iters[0] = iterations used.  n_iterations < 0 means "tolerance mode, cap 200".
 * ------------------------------------------------------------------------------------------ */
int impflow_sn_power_iter(const float* W, float* u, float* v, float* sigma, int* iters, int out_f,
                          int in_f, int n_iterations, float atol, float rtol, void* stream);
/* The same for n dense layers in ONE launch (one CTA per layer): descs is a DEVICE array of n descriptors; every layer
 * runs with the same n_iterations / atol / rtol; max_out / max_in bound the shared memory.  update_lipschitz refreshes
 * all dense layers of a model this way (train_img.py:786-792 loops over them). */
typedef struct {
  const float* W;   /* (out_f, in_f) row-major */
  float* u;         /* (out_f) in / out */
  float* v;         /* (in_f) in / out */
  float* sigma;     /* 1 float out */
  int* iters;       /* 1 int out (may be NULL) */
  int out_f, in_f;
} impflow_sn_desc;
int impflow_sn_power_iter_batch(const impflow_sn_desc* descs, int n, int max_out, int max_in, int n_iterations,
                                float atol, float rtol, void* stream);

/* The same power iteration for a 3x3 / stride 1 / pad 1 convolution acting on ONE H x W image — replaces the
 * host loop of mixed_lipschitz.py:328-386 (_compute_weight_kxk: 1-sample conv2d / conv_transpose2d,
 * normalisations and a host-synchronising tolerance test per iteration) with ONE cooperative launch.
 * W is [Cout][Cin][3][3]; u (Cout*H*W) and v (Cin*H*W) are flat CHW vectors updated in place;
 * sigma[0] = <u, conv(v)>; iters[0] = iterations used; n_iterations < 0 = tolerance mode (cap 200).
 * D (optional, W's shape) receives d sigma / d W at the final (u, v) — the correlation of u with the patches
 * of v that the gradient of the rescaled weight needs.
 * `ws` holds impflow_sn_conv_workspace_floats() floats; that function returns 0 (and the solver -2) when the
 * narrow side of the layer does not fit in shared memory (the caller then keeps its own loop). */
size_t impflow_sn_conv_workspace_floats(int Cout, int Cin, int H, int W);
/* CTAs one 3x3 power-iteration launch spreads its wide channels over (default 32, so that the independent layers of
 * update_lipschitz run side by side; 128 = the widest the cooperative launch allows).  Returns the previous value;
 * query impflow_sn_conv_workspace_floats again after changing it. */
int impflow_sn_conv_set_ctas(int ctas);
int impflow_sn_power_iter_conv3x3(const float* W, float* u, float* v, float* sigma, int* iters, int Cout, int Cin,
                                  int H, int Wd, int n_iterations, float atol, float rtol, float* ws, float* D,
                                  void* stream);

/* Soft spectral rescale with sigma on the device: out = W / max(1, sigma[0]/coeff), scale_out[0] =
 * sigma[0] (mixed_lipschitz.py:125-131), and its gradient chain with D = d sigma / d W (sigma = <W,D>
 * is linear in W; u, v constant):  out = s*G + gw_dot[0] * ds/dsigma * D,  gw_dot = <G, W>. */
/* One launch per layer and optimiser step: the rescaled weight W / max(1, sigma[0]/coeff) written in every
 * layout the branch kernels consume — forward and transposed GEMM forms (K zero-padded to fwd_k / bwd_k) as
 * fp32 and, when the plane pointers are given, tf32 hi/lo planes.  kind 0: linear / 1x1 (fwd (cout, fwd_k),
 * bwd (cin, bwd_k)); kind 1: 3x3 with cin <= cout (fwd (cout, 9cin->fwd_k), bwd (9cin, bwd_k));
 * kind 2: 3x3 with cin > cout (fwd (9cout, fwd_k), bwd (cin, 9cout->bwd_k), taps flipped).  Replaces the
 * permute / flip / pad / split sequence of the host (branch_program._prep). */
int impflow_prep_weights(const float* W, const float* sigma, float coeff, int kind, int cout, int cin, float* fwd,
                         float* fwd_hi, float* fwd_lo, int fwd_rows, int fwd_k, float* bwd, float* bwd_hi,
                         float* bwd_lo, int bwd_rows, int bwd_k, void* stream);
int impflow_sn_scale(const float* W, const float* sigma, float coeff, float* out, float* scale_out, long long n,
                     void* stream);
int impflow_sn_scale_grad(const float* G, const float* D, const float* sigma, const float* gw_dot, float coeff,
                          float* out, long long n, void* stream);
/* Same chain, reading dL/dW_eff straight from the GEMM layout the weight-gradient kernels produce (the fwd side of
 * impflow_prep_weights: kind 0 [cout][cin], 1 [cout][(ky,kx,cin)], 2 [(2-ky,2-kx,cout)][cin]; row stride ldw) and
 * writing the module's weight layout [cout][cin][3][3]: replaces the flip / permute / contiguous copies and the
 * separate <G, W> reduction (mixed_lipschitz.py:125-131 backward).  ws: 1024 floats. */
int impflow_sn_scale_grad_layout(const float* Wbar, long long ldw, const float* W, const float* D, const float* sigma,
                                 float coeff, int kind, int cout, int cin, float* out, float* ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IMPFLOW_B200_H */
