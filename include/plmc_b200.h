/*
 * plmc_b200.h -- C ABI of libplmc_b200.so, the sm_100a (B200) engine behind the
 * projected-LMC marginal-likelihood / prediction path.
 *
 * The reference (QWERTY6191/projected-lmc) has no FFI: its hot path is Python
 * that reaches torch/gpytorch/linear_operator kernels.  Each entry point below
 * names the reference call site (file:line under the reference checkout) whose
 * arithmetic it replaces; INTEGRATION.md shows the ctypes binding.
 *
 * Contract (SURVEY.md section 8b):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     the parameter name ends in _host;
 *   - the caller owns every buffer, including workspaces; the library never
 *     allocates, frees or synchronises; all work is ordered on `stream`
 *     (a cudaStream_t passed as void*);
 *   - return value: 0 ok, -1 bad argument, -2 launch failure.  Numerical
 *     failure (non-PD matrix) is reported LAPACK-style in a device `info`
 *     array, never through the return code;
 *   - re-entrant: every numerical setting is a per-call argument (plmc_gemm_cfg).
 *     The only process-wide state is (a) per-device one-time function attributes,
 *     (b) the atomic launch counters behind plmc_stats_*, (c) the DIAGNOSTIC
 *     switches plmc_trace_enable / plmc_ozaki_debug, which must not be toggled
 *     while other threads are inside the library.  Calls on different streams,
 *     from different threads, with different configurations and on different
 *     devices (cudaSetDevice to the device that owns the buffers first) may run
 *     concurrently as long as their buffers, including the plane scratch of
 *     plmc_gemm_cfg, are distinct;
 *   - FP64 throughout; matrices row-major; "npad" = n rounded up to 128.
 */
#ifndef PLMC_B200_H
#define PLMC_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define PLMC_KERNEL_RBF 0      /* exp(-s/2)                               */
#define PLMC_KERNEL_MATERN52 1 /* (1+sqrt5 r+5/3 r^2) exp(-sqrt5 r)       */
#define PLMC_KERNEL_MATERN32 2 /* (1+sqrt3 r) exp(-sqrt3 r)               */
#define PLMC_KERNEL_MATERN12 3 /* exp(-r)                                 */
#define PLMC_KERNEL_RQ 4       /* (1+s/(2 alpha))^-alpha, alpha per latent: gpytorch RQKernel */

/* Kernels with a shape parameter (PLMC_KERNEL_RQ: alpha) are reached through the ...2 entry points, which take it
 * as `shape` ([q], device, one value per latent) and return its gradient in `g_shape` ([q], may be NULL).  They
 * return PLMC_ERR_BADARG for RQ with shape == NULL, for a non-NULL shape with kernels 0-3 and for g_shape without a
 * shape.  The entry points without the 2 are these with shape = g_shape = NULL, result for result.              */

/* ---- arithmetic of the large GEMMs of the factorisation layer (per call) ----------------------
 * FP64 matrix products with M, N and K all >= min_dim and M*N*K >= min_mnk can be computed on the tcgen05 INT8
 * tensor path instead of the FP64 DMMA units (B200 has no FP64 kind on tcgen05):
 *   PLMC_GEMM_INT8_DIGITS  operands split into `precision` (1..7) signed 8-bit digit planes, 8p-1 bits
 *                          relative to the row/column maximum, p(p+1)/2 INT8 products (csrc/ozaki.cu);
 *   PLMC_GEMM_INT8_RNS     operands scaled to integers and reduced modulo `precision` (8..18) pairwise
 *                          coprime moduli <= 256; ONE INT8 product per modulus, exact integer result by
 *                          the Chinese remainder theorem (csrc/ozaki2.cu).  16 moduli = 55 bits for
 *                          K <= 16384 (plmc_rns_bits gives the bits for any K).
 * A NULL cfg (or mode PLMC_GEMM_FP64) is pure FP64 arithmetic.  `ws` is caller-owned DEVICE scratch
 * for the operand planes; a product that does not fit is processed in pieces (RNS) or falls back to
 * the FP64 kernel (digits).  Two concurrent calls must not share `ws`.                            */
#define PLMC_GEMM_FP64 0
#define PLMC_GEMM_INT8_DIGITS 1
#define PLMC_GEMM_INT8_RNS 2
#define PLMC_GEMM_FLAG_SINGLE_CTA 1 /* RNS: 128x256 single-CTA tiles instead of CTA pairs (diagnostics) */
#define PLMC_GEMM_FLAG_LEAF_SOLVES 2 /* RNS: the panel solves of potrf recurse to the 128-leaves instead of multiplying
                                        by the explicit inverses of the diagonal 2048-blocks (diagnostics, A/B timing) */
#define PLMC_GEMM_FLAG_NO_TRI 4     /* RNS: triangular multiplies (trtri / lauum / trmm) always take the recursion with
                                       dense 512-leaves instead of one launch set over the nonzero k-tiles (A/B timing) */
typedef struct plmc_gemm_cfg {
    void* ws;
    long long ws_bytes;
    int mode;
    int precision;
    int min_dim; /* >= 128 */
    int flags;
    /* mode PLMC_GEMM_INT8_RNS only: the residue scheme pays a fixed cost per output element (residues out,
     * reconstruction in), so products with a short inner dimension or little work run on digit planes instead:
     * K < rns_min_k or M*N*K < rns_min_mnk -> PLMC_GEMM_INT8_DIGITS with alt_precision planes (0: always RNS). */
    int alt_precision;
    int rns_min_k;
    long long rns_min_mnk;
    /* products with M*N*K below min_mnk stay on the FP64 kernel whatever their dimensions (0: no work floor):
     * with min_dim = 128 this sends the tall-skinny leaf applications of the triangular solves (m x 128 x 128,
     * m large) to the tensor path and keeps the tiny ones off it. */
    long long min_mnk;
} plmc_gemm_cfg;

int plmc_version(void);
/* optional: opt in to >48 KB dynamic shared memory on the current device (done lazily otherwise) */
int plmc_init(void);
/* host-side launch statistics since the last reset: kernels launched by this
 * library, GEMM launches among them, and their algorithmic FLOPs (2*M*N*K over the
 * tiles actually computed).  Outputs are HOST pointers (may be NULL).            */
int plmc_stats_reset(void);
/* account for kernels launched outside the library's own launch sites: a caller that replays a CUDA graph captured
 * over library calls adds the number of kernel nodes per replay */
int plmc_stats_add(long long launches);
int plmc_stats_get(long long* launches_host, long long* gemm_launches_host, double* gemm_flops_host);
/* diagnostics: with tracing on, every GEMM of the factorisation layer is bracketed by CUDA events;
 * plmc_trace_report synchronises the device and prints time and FLOP rate per GEMM shape to stderr. */
int plmc_trace_enable(int on);
int plmc_trace_report(void);
/* npad for a problem of order n (multiple of 128) */
long long plmc_npad(long long n);
/* bytes of the side buffer `dinv` of the factorisation calls for `batch` matrices of order npad: the 128x128
 * inverses of the diagonal Cholesky leaves (written by potrf, read by every solve) followed by ceil(npad/512)
 * slots of 512x512 for zero-padded dense copies of diagonal blocks (scratch of trtri / lauum / potri) and
 * (npad > 2048) ceil(npad/2048) slots of 2048x2048 for the explicit inverses of the diagonal 2048-blocks of L that
 * potrf keeps for its own panel solves in residue mode.                                                                */
long long plmc_dinv_bytes(long long npad, int batch);

/* ---- (1) projection: ProjectedGPModel.project_data, projected_lmc.py:1014-1021
 * TY[l, i] = sum_t T[t, l] * Y[i, t]   (T = projection_matrix(), :1003-1012)
 * Y [n, p] row-major, T [p, q] row-major, TY [q, ldty] (ldty >= n).            */
int plmc_project_fwd(const double* Y, const double* T, double* TY, long long n, int p, int q, long long ldty,
                     void* stream);
/* dT[t, l] = sum_i Y[i, t] * G[l, i]  (autograd of the matmuls at :1016-1019).
 * partial: workspace of plmc_project_bwd_ws(n,p,q) bytes.                       */
long long plmc_project_bwd_ws(long long n, int p, int q);
int plmc_project_bwd(const double* Y, const double* G, long long ldg, double* dT, double* partial, long long n,
                     int p, int q, void* stream);

/* ---- (2) Gram build: handle_covar_ kernels, projected_lmc.py:151-167, evaluated
 * at :1201; gpytorch sq_dist semantics (centre by column mean, expansion,
 * clamp_min 0), ScaleKernel and the GaussianLikelihood diagonal (:1200).       */
/* host-only helper (HOST pointers, no device work): k(s) and dk/ds of PLMC_KERNEL_* evaluated by the same source
 * the device kernels compile (csrc/kernel_math.cuh: hand-written exp / sqrt), for CPU-side accuracy tests. */
int plmc_kernel_profile_host(int kernel_id, const double* s_host, long long n, double* k_host, double* dk_host);
/* host-only helper: sqrt(s) and 1/sqrt(s) as the Cholesky leaf computes its pivots (one coupled Goldschmidt
 * iteration, csrc/kernel_math.cuh), for CPU-side accuracy tests; s <= 0 gives NaN for both. */
int plmc_sqrt_reciprocal_host(const double* s_host, long long n, double* root_host, double* inv_host);
/* host-only helper: k(s), dk/ds and dk/dshape (gpytorch RQKernel.forward and its autograd; 0 for kernels 0-3) with
 * shape_host[i] the shape parameter of entry i (NULL for kernels 0-3). */
int plmc_kernel_profile2_host(int kernel_id, const double* s_host, const double* shape_host, long long n,
                              double* k_host, double* dk_host, double* dshape_host);
/* host-only helper: log(1 + x), x >= 0, as the RQ kernel computes it on the device (torch.log1p in RQKernel) */
int plmc_log1p_host(const double* x_host, long long n, double* out_host);
/* xmean[k] = mean_i X[i,k] */
int plmc_col_mean(const double* X, long long n, int d, double* xmean, void* stream);
/* Z[l, i, k] = (X[i,k]-xmean[k]) / ell[l,k], zero padded to [q, rows_pad, dpad];
 * zn[l, i] = sum_k Z^2.  dpad % 4 == 0, rows_pad >= n.                          */
int plmc_scale_inputs(const double* X, const double* xmean, const double* ell, double* Z, double* zn, long long n,
                      int d, int dpad, long long rows_pad, int q, void* stream);
/* K[l] (lower 128-tiles of a [npad, ld] matrix) = os[l]*k(s_ij) + diag_add[l]*I,
 * identity in the padding.  os may be NULL (no ScaleKernel).  accumulate != 0: K[l] += os[l]*k(s_ij)
 * (a further component of an additive kernel, handle_covar_ `decomp`, projected_lmc.py:151-167; the
 * diagonal term and the padding belong to the first component).                                    */
int plmc_gram(const double* Z, const double* zn, int kernel_id, const double* os, const double* diag_add, double* K,
              long long ld, long long stride, long long n, long long npad, int dpad, int q, int accumulate,
              void* stream);
/* Kx[l, i, j] = os[l]*k(train_i, test_j): [q, npad, ldx] with ldx >= mt, mt%128==0;
 * rows >= n are zero.                                                            */
int plmc_cross_gram(const double* Ztrain, const double* zntrain, const double* Ztest, const double* zntest,
                    int kernel_id, const double* os, double* Kx, long long ldx, long long stride, long long n,
                    long long npad, long long mt_rows_pad, long long mt, int dpad, int q, int accumulate,
                    void* stream);
/* plmc_gram / plmc_cross_gram with the kernel's shape parameter (RQKernel.forward under ScaleKernel, reached from
 * projected_lmc.py:151-167 with kernel_type=RQKernel; the test-point block of exact_prediction likewise). */
int plmc_gram2(const double* Z, const double* zn, int kernel_id, const double* os, const double* shape,
               const double* diag_add, double* K, long long ld, long long stride, long long n, long long npad, int dpad,
               int q, int accumulate, void* stream);
int plmc_cross_gram2(const double* Ztrain, const double* zntrain, const double* Ztest, const double* zntest,
                     int kernel_id, const double* os, const double* shape, double* Kx, long long ldx, long long stride,
                     long long n, long long npad, long long mt_rows_pad, long long mt, int dpad, int q, int accumulate,
                     void* stream);

/* ---- adjoint of the cross-Gram block (inducing-point / SGPR variant: ExactGPModel(n_inducing_points=m),
 * projected_lmc.py:302-303 -> gpytorch InducingPointKernel).  Zr [q, rows_pad_r, dpad] / Zc [q, rows_pad_c, dpad]
 * are the scaled row (inducing) and column (data) points as produced by plmc_scale_inputs, G [q, nr, ldg] the
 * cotangent of K[l,i,j] = os[l] k(|zr_i - zc_j|^2).  Outputs: g_ell [q, d], g_os [q] (may be NULL),
 * g_rows [nr, d] = gradient w.r.t. the UNscaled row points summed over the latents.  partial: workspace of
 * plmc_cross_gram_bwd_ws(nr, nc, d, q) bytes.  Deterministic (fixed-order reductions, no atomics).          */
long long plmc_cross_gram_bwd_ws(long long nr, long long nc, int d, int q);
int plmc_cross_gram_bwd(const double* Zr, long long rows_pad_r, const double* Zc, long long rows_pad_c, const double* G,
                        long long ldg, long long strideG, int kernel_id, const double* os, const double* ell,
                        double* g_ell, double* g_os, double* g_rows, double* partial, long long nr, long long nc, int d,
                        int dpad, int q, void* stream);
/* with the kernel's shape parameter (autograd of RQKernel.forward inside InducingPointKernel): g_shape [q] = dL/dshape;
 * partial: plmc_cross_gram_bwd_ws2(nr, nc, d, q, kernel_id) bytes */
long long plmc_cross_gram_bwd_ws2(long long nr, long long nc, int d, int q, int kernel_id);
int plmc_cross_gram_bwd2(const double* Zr, long long rows_pad_r, const double* Zc, long long rows_pad_c,
                         const double* G, long long ldg, long long strideG, int kernel_id, const double* os,
                         const double* shape, const double* ell, double* g_ell, double* g_os, double* g_shape,
                         double* g_rows, double* partial, long long nr, long long nc, int d, int dpad, int q,
                         void* stream);

/* ---- (3) factorisation: MultivariateNormal.log_prob -> psd_safe_cholesky,
 * triangular solve, logdet (gpytorch; reached from projected_lmc.py:1201).     */
int plmc_potrf_batched(double* K, long long ld, long long stride, long long npad, int batch, double* dinv, int* info,
                       const plmc_gemm_cfg* cfg, void* stream);
/* op: 0 X L^T = aB (B m x npad) | 1 X L = aB | 2 L X = aB (B npad x m) | 3 L^T X = aB ; m % 128 == 0 */
int plmc_trsm_batched(int op, const double* L, long long ld, long long stride, long long npad, int batch,
                      const double* dinv, double* B, long long ldb, long long strideb, long long m, double alpha,
                      const plmc_gemm_cfg* cfg, void* stream);
/* Triangular MULTIPLY in place with a LOWER triangular X [npad, npad] (its strict upper part is not read):
 *   op 1: B := alpha B X  (B [m, npad])  |  op 2: B := alpha X B  |  op 3: B := X^T B (alpha = 1)   (B [npad, m]),
 * m % 128 == 0: the products the explicit inverse is built from (csrc/linalg.cu).  In residue mode a large enough
 * product is ONE launch set whose INT8 GEMM visits only the k-tiles that can be nonzero (csrc/ozaki2.cu rns_trmm);
 * otherwise a recursion with dense 512-leaves.  With X = inv(L) from plmc_trtri_batched, op 2 replaces the
 * triangular solve of the predictive variance (gpytorch exact_predictive_covar, reached from projected_lmc.py:1134)
 * at GEMM speed.  dinv: the side buffer of the factorisation calls; its dense-block scratch part is overwritten
 * with copies of X's diagonal blocks.  Other ops: PLMC_ERR_BADARG.                                              */
int plmc_trmm_batched(int op, const double* X, long long ld, long long stride, long long npad, int batch, double* dinv,
                      double* B, long long ldb, long long strideb, long long m, double alpha,
                      const plmc_gemm_cfg* cfg, void* stream);
/* rhs [batch, npad, 128] workspace (the first npad entries per member are used).
 * Fills z = L^-1 y, alpha = L^-T z (both [batch, ldv]), quad[b] = |z|^2,
 * logdet[b] = 2 sum log L_ii.  Two HBM-bound block substitutions: every tile of
 * the lower triangle is read once per solve (csrc/trsv.cu).                     */
int plmc_solve_logdet(const double* L, long long ld, long long stride, long long n, long long npad, int batch,
                      const double* dinv, const double* y, long long ldy, double* rhs, double* z, double* alpha,
                      long long ldv, double* quad, double* logdet, void* stream);
/* L -> inv(L) (lower) in place */
int plmc_trtri_batched(double* L, long long ld, long long stride, long long npad, int batch, double* dinv,
                       const plmc_gemm_cfg* cfg, void* stream);
/* L -> lower(L^T L) in place (dinv: only its dense-block scratch part is used, and overwritten) */
int plmc_lauum_batched(double* L, long long ld, long long stride, long long npad, int batch, double* dinv,
                       const plmc_gemm_cfg* cfg, void* stream);
/* L -> lower(K^-1) in place = trtri + lauum */
int plmc_potri_batched(double* L, long long ld, long long stride, long long npad, int batch, double* dinv,
                       const plmc_gemm_cfg* cfg, void* stream);

/* ---- (4) fused backward: autograd of log_prob through the kernel
 * (experiments.py:270 loss.backward()).  With W = 1/2 (alpha alpha^T - K^-1):
 *   g_noise[l] = tr W ; g_os[l] = sum W o k ; g_ell[l,k] = d lp / d ell[l,k].
 * Kinv: lower tiles of K^-1; Z, zn: scaled inputs and their squared norms (plmc_scale_inputs); partial: workspace
 * of plmc_grad_ws(...) bytes.  d <= 24: both contractions (distances, A Z) on the FP64 tensor cores; 24 < d <= 44:
 * direct-difference kernel; wider inputs: PLMC_ERR_BADARG (split the kernel into additive `decomp` groups).      */
long long plmc_grad_ws(long long npad, int d, int q);
/* diagnostics (process-wide, like plmc_trace_enable): direct != 0 forces the direct-difference sweep kernel that
 * otherwise only serves inputs of more than 24 dimensions; 0 restores the default (GEMM form on DMMA for d <= 24) */
int plmc_sweep_debug(int direct);
int plmc_grad_sweep(const double* Kinv, long long ld, long long stride, const double* alpha, long long lda_vec,
                    const double* Z, const double* zn, const double* ell, int kernel_id, const double* os,
                    double* g_ell, double* g_os, double* g_noise, double* partial, long long n, long long npad, int d,
                    int dpad, int q, void* stream);
/* with the kernel's shape parameter (loss.backward() through RQKernel.forward, experiments.py:270):
 * g_shape[l] = sum W o dk/dshape, accumulated beside g_os in the same fixed order; partial: plmc_grad_ws2(npad, d, q,
 * kernel_id) bytes */
long long plmc_grad_ws2(long long npad, int d, int q, int kernel_id);
int plmc_grad_sweep2(const double* Kinv, long long ld, long long stride, const double* alpha, long long lda_vec,
                     const double* Z, const double* zn, const double* ell, int kernel_id, const double* os,
                     const double* shape, double* g_ell, double* g_os, double* g_noise, double* g_shape,
                     double* partial, long long n, long long npad, int d, int dpad, int q, void* stream);

/* ---- prediction: eval ProjectedGPModel.__call__, projected_lmc.py:1121-1155 +
 * gpytorch exact_prediction.  Given V = L^-1 Kx (trsm op 2 applied to Kx):
 *   lat_mean[l, j] = sum_i alpha[l,i] Kx[l,i,j]  (call before the trsm)
 *   lat_var [l, j] = os[l]*k(0) - sum_i V[l,i,j]^2                              */
int plmc_latent_mean(const double* Kx, long long ldx, long long stride, const double* alpha, long long lda_vec,
                     double* lat_mean, long long ldm, long long n, long long mt, int q, void* stream);
int plmc_latent_var(const double* V, long long ldx, long long stride, const double* os, double* lat_var,
                    long long ldm, long long npad, long long mt, int q, void* stream);
/* mean[j,t] (+)= sum_l lat_mean[l,j] H[l,t]; var[j,t] (+)= sum_l lat_var[l,j] H[l,t]^2
 * (+ var_add[t] when accumulate == 0).  H [q, p] row-major (= lmc_coefficients()). */
int plmc_mix_tasks(const double* lat_mean, const double* lat_var, long long ldm, const double* H,
                   const double* var_add, double* mean, double* var, long long mt, int p, int q, int accumulate,
                   void* stream);

/* ---- joint predictive covariance and posterior draws (the full MultitaskMultivariateNormal of the eval branch,
 * projected_lmc.py:1149-1155: covariance sum_l C_l (x) h_l h_l^T + eps I, + I (x) F F^T after full_likelihood).
 * Latent posterior covariance C_l = K**_l - V_l^T V_l:  K**_l from plmc_gram on the scaled test points (diag_add 0),
 * then  lower(C[l]) = alpha A[l]^T A[l] + beta C[l]  with A[l] = V_l [k, ldA] row-major (k rows, n columns),
 * C [batch, n, ldc]; n % 128 == 0, k % 128 == 0.  One product per call, routed like the products of the factorisation
 * (plmc_gemm_cfg: residue planes, digit planes or FP64 DMMA), the operand converted once (SYRK).                   */
int plmc_syrk_batched(const double* A, long long lda, long long strideA, double* C, long long ldc, long long strideC,
                      long long n, long long k, double alpha, double beta, int batch, const plmc_gemm_cfg* cfg,
                      void* stream);
/* T[(i,t),(j,s)] = sum_l C[l,i,j] H[l,t] H[l,s] + [i == j] S[t,s]   (point-major, task-minor; N = ns p)
 * from the entries i >= j of C [q, >= ns, ldc] only; H [q, p] row-major; S [p, p] symmetric (T is then exactly
 * symmetric).  tiled 0: T dense [N, ldt], ldt >= N;  tiled 1: the lower 128-tiles of a [npad(N), ldt] matrix with
 * identity padding (the operand of plmc_potrf_batched, batch 1).  Writes 8 N^2 (about 4 npad(N)^2) bytes.           */
int plmc_task_covariance(const double* C, long long ldc, long long stride, const double* H, const double* S,
                         double* T, long long ldt, long long ns, int p, int q, int tiled, void* stream);
/* out[s, j, t] = mean[j, t] + sum_l G[l, j, s] H[l, t] + sum_u E[s, j, u] R[t, u]
 * mean [ns, p]; G [q, >= ns, ldg] latent draws (e.g. chol(C_l) eps_l from plmc_trmm_batched op 2, ldg >= S);
 * H [q, p]; E [S, ns, p] standard normals; R [p, p] a root of the task-level noise (R R^T = S above);
 * out [S, ns, p].  Each sample is written once.                                                                   */
int plmc_mix_samples(const double* mean, const double* G, long long ldg, long long strideg, const double* H,
                     const double* E, const double* R, double* out, long long ns, long long S, int p, int q,
                     void* stream);

/* ---- generic FP64 tensor-core GEMM (exposed for tests and roofline runs)
 * layout bit0: B(k,n) n-contiguous, bit1: A(m,k) m-contiguous (see gemm_dmma.cuh) */
int plmc_gemm(int layout, const double* A, long long lda, long long sA, const double* B, long long ldb, long long sB,
              double* C, long long ldc, long long sC, int M, int N, int K, double alpha, double beta, int lower,
              int triA, int triB, int batch, void* stream);

/* ---- FP64 GEMM on the tcgen05 INT8 tensor path (Ozaki splitting; csrc/ozaki.cu):
 * C = alpha op(A) op(B) + beta C for ONE matrix, M%128==0, N%128==0, K%32==0.
 * `slices` (1..7) signed 8-bit planes (balanced base-256 digits) per operand -> 8*slices-1
 * mantissa bits relative to the largest entry of each row of op(A) / column of op(B); 7 slices
 * reproduce a DGEMM to its own rounding level.  same_operand != 0: op(B)^T is op(A) (SYRK),
 * sliced once.  ws: plmc_ozaki_ws_bytes(...) bytes of scratch.                                */
long long plmc_ozaki_ws_bytes(int M, int N, int K, int slices, int same_operand);
/* diagnostics: with a device buffer of 64 x 8 int64 set, CTA 0 of every later INT8 GEMM launch records
 * clock64 stamps per tile (0 MMA start, 1 last MMA issued, 2 accumulators complete, 3 TMEM drained,
 * 4 C written, 5/6 first/last copy issued); NULL switches it off.                                  */
int plmc_ozaki_debug(long long* stamps);
int plmc_ozaki_gemm(int layout, const double* A, long long lda, const double* B, long long ldb, double* C,
                    long long ldc, int M, int N, int K, double alpha, double beta, int lower, int slices,
                    int same_operand, void* ws, long long ws_bytes, void* stream);

/* ---- FP64 GEMM on the tcgen05 INT8 tensor path, residue-number-system scheme (csrc/ozaki2.cu):
 * C = alpha op(A) op(B) + beta C for ONE matrix; M, N, K multiples of 128.  `moduli` (8..18) INT8
 * products (one per modulus, CTA-pair tcgen05.mma.cta_group::2 kernel) + Chinese-remainder
 * reconstruction in FP64.  plmc_rns_bits: operand bits relative to the row (column) maximum for an
 * inner dimension K (2 K 4^bits < product of the moduli).  ws: >= plmc_rns_ws_bytes(...) gives one
 * pass; a smaller scratch makes the call split the product.  flags: PLMC_GEMM_FLAG_*.            */
int plmc_rns_bits(int moduli, int K);
long long plmc_rns_ws_bytes(int M, int N, int K, int moduli, int same_operand, int lower);
/* host-only helper (no device work): moduli p_i, the leading 40 bits H_i and the tail L_i of
 * ((P/p_i)^-1 mod p_i) / p_i, pscale = P 2^(-2 bits) and the operand bits for (moduli, K).        */
int plmc_rns_constants(int moduli, int K, int* moduli_out, double* H, double* L, double* pscale, int* bits);
int plmc_rns_gemm(int layout, const double* A, long long lda, const double* B, long long ldb, double* C,
                  long long ldc, int M, int N, int K, double alpha, double beta, int lower, int moduli,
                  int same_operand, void* ws, long long ws_bytes, int flags, void* stream);

/* ---- roofline denominators (time with CUDA events on `stream`) */
int plmc_peak_dmma(int blocks, int threads, long long iters, double* scratch, void* stream);
int plmc_peak_dfma(int blocks, int threads, long long iters, double* scratch, void* stream);
int plmc_peak_copy(const double* src, double* dst, long long n, void* stream);
/* INT8 tensor-pipe peak: every SM (cta_group 1) or SM pair (cta_group 2) issues iters x 4
 * tcgen05.mma.kind::i8 of 128(256) x 256 x 32 on shared-memory-resident operands; *ops_host (HOST
 * pointer) receives the INT8 operations (2 per MAC) of the launch.  scratch is unused.          */
int plmc_peak_i8(long long iters, int cta_group, void* scratch, double* ops_host, void* stream);
/* even warps run the DMMA loop (iters_mma x 16 x 512 FLOP per warp), odd warps the DFMA loop
 * (iters_fma x 16 x 2 FLOP per thread): shows that on B200 the two share one FP64 datapath
 * (measured sum 35-36 TFLOP/s for every mix), i.e. 37 TFLOP/s is the FP64 roof.          */
int plmc_peak_mixed(int blocks, int threads, long long iters_mma, long long iters_fma, double* scratch,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif
