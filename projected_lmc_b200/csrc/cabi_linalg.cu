// C ABI: factorisation layer (see include/plmc_b200.h for the contract).
#include "linalg.cuh"

using namespace plmc;

namespace plmc {

// quad[b] = sum z_i^2 ; logdet[b] = 2 sum log L_ii   (fixed-order reduction)
__global__ void __launch_bounds__(1024) quad_logdet_kernel(const double* __restrict__ z, long long ldv,
                                                            const double* __restrict__ L, long long ld,
                                                            long long stride, long long n, double* __restrict__ quad,
                                                            double* __restrict__ logdet) {
    __shared__ double sh[32];
    const int b = blockIdx.x;
    const double* Z = z + (long long)b * ldv;
    const double* Lb = L + (long long)b * stride;
    double sq = 0.0, sl = 0.0;
    for (long long i = threadIdx.x; i < n; i += 1024) {
        const double v = Z[i];
        sq += v * v;
        sl += log(Lb[i * ld + i]);
    }
    sq = block_sum<1024>(sq, sh);
    sl = block_sum<1024>(sl, sh);
    if (threadIdx.x == 0) {
        quad[b] = sq;
        logdet[b] = 2.0 * sl;
    }
}

}  // namespace plmc

#include "plmc_b200.h"

// The arithmetic of the large GEMMs is a PER-CALL argument (plmc_gemm_cfg): no process-wide setting.
// Returns false for an inconsistent configuration.
static bool make_ctx(LaCtx& cx, cudaStream_t st, int batch, const plmc_gemm_cfg* cfg) {
    cx = LaCtx{st, batch, 0};
    if (!cfg || cfg->mode == PLMC_GEMM_FP64) return true;
    if (cfg->mode == PLMC_GEMM_INT8_DIGITS) {
        if (cfg->precision < 1 || cfg->precision > 7) return false;
    } else if (cfg->mode == PLMC_GEMM_INT8_RNS) {
        if (cfg->precision < 8 || cfg->precision > 18 || cfg->alt_precision < 0 || cfg->alt_precision > 7) return false;
    } else {
        return false;
    }
    if (!cfg->ws || cfg->ws_bytes <= 0 || cfg->min_dim < 128) return false;
    cx.oz_ws = cfg->ws;
    cx.oz_bytes = cfg->ws_bytes;
    cx.oz_mode = cfg->mode;
    cx.oz_prec = cfg->precision;
    cx.oz_min = cfg->min_dim;
    cx.oz_min_mnk = cfg->min_mnk;
    cx.oz_flags = cfg->flags;
    if (cfg->mode == PLMC_GEMM_INT8_RNS) {
        cx.oz_alt = cfg->alt_precision;
        cx.oz_rns_min_k = cfg->rns_min_k;
        cx.oz_rns_min_mnk = cfg->rns_min_mnk;
    }
    return true;
}

extern "C" {

int plmc_version(void) { return 100; }

int plmc_trace_enable(int on) {
    trace_enable(on != 0);
    return PLMC_OK;
}
int plmc_trace_report(void) {
    trace_report();
    return PLMC_OK;
}

int plmc_init(void) { return gemm_init_attrs(); }

int plmc_stats_reset(void) {
    stats_reset();
    return PLMC_OK;
}

int plmc_stats_add(long long launches) {
    note_launch(launches);
    return PLMC_OK;
}

int plmc_stats_get(long long* launches_host, long long* gemm_launches_host, double* gemm_flops_host) {
    stats_get(launches_host, gemm_launches_host, gemm_flops_host);
    return PLMC_OK;
}

long long plmc_npad(long long n) { return ((n + 127) / 128) * 128; }

long long plmc_dinv_bytes(long long npad, int batch) { return dinv_elems(npad) * 8 * (long long)batch; }

int plmc_gemm(int layout, const double* A, long long lda, long long sA, const double* B, long long ldb, long long sB,
              double* C, long long ldc, long long sC, int M, int N, int K, double alpha, double beta, int lower,
              int triA, int triB, int batch, void* stream) {
    if (!A || !B || !C) return PLMC_ERR_BADARG;
    GemmArgs g;
    g.A = A; g.B = B; g.C = C;
    g.lda = lda; g.ldb = ldb; g.ldc = ldc;
    g.sA = sA; g.sB = sB; g.sC = sC;
    g.M = M; g.N = N; g.K = K;
    g.alpha = alpha; g.beta = beta;
    g.lower = lower; g.triA = triA; g.triB = triB;
    const bool aKC = !(layout & 2), bKC = !(layout & 1);
    return gemm_launch(aKC, bKC, g, batch, (cudaStream_t)stream);
}

static bool bad_mat(const void* p, long long ld, long long npad, int batch) {
    return !p || npad <= 0 || (npad % 128) || ld < npad || (ld & 1) || batch <= 0 || batch > 65535 ||
           npad > 2147483647LL;
}

int plmc_potrf_batched(double* K, long long ld, long long stride, long long npad, int batch, double* dinv, int* info,
                       const plmc_gemm_cfg* cfg, void* stream) {
    if (bad_mat(K, ld, npad, batch) || !dinv || !info) return PLMC_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    LaCtx cx;
    if (!make_ctx(cx, st, batch, cfg)) return PLMC_ERR_BADARG;
    if (cudaMemsetAsync(info, 0, sizeof(int) * batch, st) != cudaSuccess) return PLMC_ERR_LAUNCH;
    potrf_lower(cx, BMat{K, ld, stride}, (int)npad, make_dinv(dinv, npad), 0, info);
    return cx.status;
}

int plmc_trsm_batched(int op, const double* L, long long ld, long long stride, long long npad, int batch,
                      const double* dinv, double* B, long long ldb, long long strideb, long long m, double alpha,
                      const plmc_gemm_cfg* cfg, void* stream) {
    if (bad_mat(L, ld, npad, batch) || !dinv || !B || m <= 0 || (m % 128) || (ldb & 1)) return PLMC_ERR_BADARG;
    LaCtx cx;
    if (!make_ctx(cx, (cudaStream_t)stream, batch, cfg)) return PLMC_ERR_BADARG;
    BMat Lm{const_cast<double*>(L), ld, stride};
    DinvBuf D = make_dinv(dinv, npad);
    BMat Bm{B, ldb, strideb};
    switch (op) {
        case 0: trsm_rlt(cx, Lm, (int)npad, D, 0, Bm, (int)m, alpha); break;
        case 1: trsm_rln(cx, Lm, (int)npad, D, 0, Bm, (int)m, alpha); break;
        case 2: trsm_lln(cx, Lm, (int)npad, D, 0, Bm, (int)m, alpha); break;
        case 3: trsm_llt(cx, Lm, (int)npad, D, 0, Bm, (int)m, alpha); break;
        default: return PLMC_ERR_BADARG;
    }
    return cx.status;
}

int plmc_trmm_batched(int op, const double* X, long long ld, long long stride, long long npad, int batch, double* dinv,
                      double* B, long long ldb, long long strideb, long long m, double alpha,
                      const plmc_gemm_cfg* cfg, void* stream) {
    if (op < 1 || op > 3 || (op == 3 && alpha != 1.0) || bad_mat(X, ld, npad, batch) || !dinv || !B || m <= 0 ||
        (m % 128) || (ldb & 1))
        return PLMC_ERR_BADARG;
    LaCtx cx;
    if (!make_ctx(cx, (cudaStream_t)stream, batch, cfg)) return PLMC_ERR_BADARG;
    trmm_lower(cx, op, BMat{const_cast<double*>(X), ld, stride}, (int)npad, make_dinv(dinv, npad), BMat{B, ldb, strideb},
               (int)m, alpha);
    return cx.status;
}

int plmc_solve_logdet(const double* L, long long ld, long long stride, long long n, long long npad, int batch,
                      const double* dinv, const double* y, long long ldy, double* rhs, double* z, double* alpha,
                      long long ldv, double* quad, double* logdet, void* stream) {
    if (bad_mat(L, ld, npad, batch) || !dinv || !y || !rhs || !z || !alpha || !quad || !logdet || n <= 0 ||
        n > npad || ldv < n || ldy < n)
        return PLMC_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    // two HBM-bound block substitutions on one vector (csrc/trsv.cu); rhs is the npad-vector workspace
    const int rc = trsv_solve(L, ld, stride, dinv, dinv_elems(npad), y, ldy, rhs, npad * 128, z, alpha, ldv, n, npad, batch, st);
    if (rc) return rc;
    quad_logdet_kernel<<<batch, 1024, 0, st>>>(z, ldv, L, ld, stride, n, quad, logdet);
    PLMC_CHECK_LAUNCH();
    note_launch(4);
    return PLMC_OK;
}

int plmc_trtri_batched(double* L, long long ld, long long stride, long long npad, int batch, double* dinv,
                       const plmc_gemm_cfg* cfg, void* stream) {
    if (bad_mat(L, ld, npad, batch) || !dinv) return PLMC_ERR_BADARG;
    LaCtx cx;
    if (!make_ctx(cx, (cudaStream_t)stream, batch, cfg)) return PLMC_ERR_BADARG;
    trtri_lower(cx, BMat{L, ld, stride}, (int)npad, make_dinv(dinv, npad), 0);
    return cx.status;
}

int plmc_lauum_batched(double* L, long long ld, long long stride, long long npad, int batch, double* dinv,
                       const plmc_gemm_cfg* cfg, void* stream) {
    if (bad_mat(L, ld, npad, batch) || !dinv) return PLMC_ERR_BADARG;
    LaCtx cx;
    if (!make_ctx(cx, (cudaStream_t)stream, batch, cfg)) return PLMC_ERR_BADARG;
    lauum_lower(cx, BMat{L, ld, stride}, (int)npad, make_dinv(dinv, npad), 0, /*fill_dense=*/true);
    return cx.status;
}

int plmc_syrk_batched(const double* A, long long lda, long long strideA, double* C, long long ldc, long long strideC,
                      long long n, long long k, double alpha, double beta, int batch, const plmc_gemm_cfg* cfg,
                      void* stream) {
    if (!A || k <= 0 || (k % 128) || k > 2147483647LL || lda < n || (lda & 1) || bad_mat(C, ldc, n, batch))
        return PLMC_ERR_BADARG;
    LaCtx cx;
    if (!make_ctx(cx, (cudaStream_t)stream, batch, cfg)) return PLMC_ERR_BADARG;
    syrk_lower(cx, BMat{const_cast<double*>(A), lda, strideA}, (int)n, (int)k, BMat{C, ldc, strideC}, alpha, beta);
    return cx.status;
}

int plmc_potri_batched(double* L, long long ld, long long stride, long long npad, int batch, double* dinv,
                       const plmc_gemm_cfg* cfg, void* stream) {
    if (bad_mat(L, ld, npad, batch) || !dinv) return PLMC_ERR_BADARG;
    LaCtx cx;
    if (!make_ctx(cx, (cudaStream_t)stream, batch, cfg)) return PLMC_ERR_BADARG;
    DinvBuf D = make_dinv(dinv, npad);
    trtri_lower(cx, BMat{L, ld, stride}, (int)npad, D, 0);
    lauum_lower(cx, BMat{L, ld, stride}, (int)npad, D, 0, /*fill_dense=*/false);   // trtri left the dense copies
    return cx.status;
}
}
