// Batched predictive mean / variance epilogues.
//
// Replaces the eval branch of ProjectedGPModel.__call__ (projected_lmc.py:1121-1155)
// and gpytorch's exact_prediction: per latent l and test point j
//   m_l[j] = k*_l(j)^T alpha_l,   v_l[j] = k_l(x*,x*) - | L_l^-1 k*_l(j) |^2
// and the task mixing  mean[j,t] = sum_l m_l[j] H[l,t],
//                      var [j,t] = sum_l v_l[j] H[l,t]^2 + eps (+ diag Sigma).
// The reference materialises the full [q, n*, n*] posterior covariance and a
// dense Kronecker sum (:1149-1153); .mean / .variance need only its diagonal,
// which is what is computed here, eagerly and tiled over the test points.  The
// joint quantities (covariance_matrix, rsample, log_prob) are computed on demand
// from the latent blocks C_l = K**_l - V_l^T V_l by csrc/joint.cu.
//
// Kx / V are [q, npad, ldx] (train row, test column); the O(n^2 n*) part is the
// TRSM (plmc_trsm_batched op 2) between the two reductions below.
#include "plmc_common.cuh"

namespace plmc {

constexpr int PR_COLS = 128;   // test columns per CTA
constexpr int PR_SPLIT = 8;    // row groups per CTA (256 threads = 32 x 8 ... see below)

// out[l, j] = base - sign * sum_i f(M[l, i, j])  with f = w_i * x (mean) or x^2 (var)
// CTA: 128 columns x 8 row-groups (1024 threads); fixed-order reduction.
template <bool SQUARE>
__global__ void __launch_bounds__(1024) col_reduce_kernel(const double* __restrict__ M, long long ldx,
                                                          long long stride, const double* __restrict__ wvec,
                                                          long long ldw, const double* __restrict__ os,
                                                          double* __restrict__ out, long long ldm, long long rows,
                                                          long long mt) {
    __shared__ double sh[PR_SPLIT][PR_COLS];
    const int l = blockIdx.z;
    const int c = threadIdx.x & (PR_COLS - 1), grp = threadIdx.x >> 7;
    const long long j = (long long)blockIdx.x * PR_COLS + c;
    const double* Ml = M + (long long)l * stride;
    const double* w = SQUARE ? nullptr : wvec + (long long)l * ldw;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (j < mt) {
        long long i = grp;
        for (; i + 3 * PR_SPLIT < rows; i += 4 * PR_SPLIT) {
            const double a0 = Ml[i * ldx + j], a1 = Ml[(i + PR_SPLIT) * ldx + j];
            const double a2 = Ml[(i + 2 * PR_SPLIT) * ldx + j], a3 = Ml[(i + 3 * PR_SPLIT) * ldx + j];
            if (SQUARE) {
                s0 = fma(a0, a0, s0); s1 = fma(a1, a1, s1); s2 = fma(a2, a2, s2); s3 = fma(a3, a3, s3);
            } else {
                s0 = fma(a0, w[i], s0); s1 = fma(a1, w[i + PR_SPLIT], s1);
                s2 = fma(a2, w[i + 2 * PR_SPLIT], s2); s3 = fma(a3, w[i + 3 * PR_SPLIT], s3);
            }
        }
        for (; i < rows; i += PR_SPLIT) {
            const double a0 = Ml[i * ldx + j];
            s0 = SQUARE ? fma(a0, a0, s0) : fma(a0, w[i], s0);
        }
    }
    sh[grp][c] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (grp == 0 && j < mt) {
        double s = 0.0;
#pragma unroll
        for (int g8 = 0; g8 < PR_SPLIT; ++g8) s += sh[g8][c];
        if (SQUARE)
            out[(long long)l * ldm + j] = (os ? os[l] : 1.0) - s;
        else
            out[(long long)l * ldm + j] = s;
    }
}

// mean[j,t] = sum_l lm[l,j] H[l,t] ; var[j,t] = sum_l lv[l,j] H[l,t]^2 + var_add[t]
constexpr int MX_J = 32, MX_T = 64, MX_L = 32;
__global__ void __launch_bounds__(256) mix_tasks_kernel(const double* __restrict__ lm, const double* __restrict__ lv,
                                                        long long ldm, const double* __restrict__ H,
                                                        const double* __restrict__ var_add, double* __restrict__ mean,
                                                        double* __restrict__ var, long long mt, int p, int q,
                                                        int accumulate) {
    __shared__ double Hs[MX_L][MX_T];
    __shared__ double ms[MX_L][MX_J + 1];
    __shared__ double vs[MX_L][MX_J + 1];
    const int tid = threadIdx.x;
    const long long j0 = (long long)blockIdx.x * MX_J;
    const int t0 = blockIdx.y * MX_T;
    const int tl = tid & (MX_T - 1), jg = tid >> 6;  // 4 row groups x 64 tasks
    double am[MX_J / 4], av[MX_J / 4];
#pragma unroll
    for (int a = 0; a < MX_J / 4; ++a) am[a] = av[a] = 0.0;

    for (int l0 = 0; l0 < q; l0 += MX_L) {
        const int lc = min(MX_L, q - l0);
        __syncthreads();
        for (int idx = tid; idx < MX_L * MX_T; idx += 256) {
            const int l = idx >> 6, t = idx & 63;
            Hs[l][t] = (l < lc && t0 + t < p) ? H[(long long)(l0 + l) * p + t0 + t] : 0.0;
        }
        for (int idx = tid; idx < MX_L * MX_J; idx += 256) {
            const int l = idx >> 5, j = idx & 31;
            const bool ok = (l < lc) && (j0 + j < mt);
            ms[l][j] = ok ? lm[(long long)(l0 + l) * ldm + j0 + j] : 0.0;
            vs[l][j] = (ok && lv) ? lv[(long long)(l0 + l) * ldm + j0 + j] : 0.0;
        }
        __syncthreads();
        for (int l = 0; l < lc; ++l) {
            const double h = Hs[l][tl];
            const double h2 = h * h;
#pragma unroll
            for (int a = 0; a < MX_J / 4; ++a) {
                am[a] = fma(ms[l][jg + 4 * a], h, am[a]);
                av[a] = fma(vs[l][jg + 4 * a], h2, av[a]);
            }
        }
    }
    const int t = t0 + tl;
    if (t < p) {
        const double va = (var_add && !accumulate) ? var_add[t] : 0.0;
#pragma unroll
        for (int a = 0; a < MX_J / 4; ++a) {
            const long long j = j0 + jg + 4 * a;
            if (j < mt) {
                const long long o = j * p + t;
                if (accumulate) {
                    mean[o] += am[a];
                    if (var) var[o] += av[a];
                } else {
                    mean[o] = am[a];
                    if (var) var[o] = av[a] + va;
                }
            }
        }
    }
}

}  // namespace plmc

using namespace plmc;

extern "C" {

int plmc_latent_mean(const double* Kx, long long ldx, long long stride, const double* alpha, long long lda_vec,
                     double* lat_mean, long long ldm, long long n, long long mt, int q, void* stream) {
    if (!Kx || !alpha || !lat_mean || n <= 0 || mt <= 0 || ldx < mt || ldm < mt || lda_vec < n || q <= 0 || q > 65535)
        return PLMC_ERR_BADARG;
    dim3 grid((unsigned)((mt + PR_COLS - 1) / PR_COLS), 1, q);
    col_reduce_kernel<false><<<grid, 1024, 0, (cudaStream_t)stream>>>(Kx, ldx, stride, alpha, lda_vec, nullptr,
                                                                      lat_mean, ldm, n, mt);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}

int plmc_latent_var(const double* V, long long ldx, long long stride, const double* os, double* lat_var,
                    long long ldm, long long npad, long long mt, int q, void* stream) {
    if (!V || !lat_var || npad <= 0 || mt <= 0 || ldx < mt || ldm < mt || q <= 0 || q > 65535)
        return PLMC_ERR_BADARG;
    dim3 grid((unsigned)((mt + PR_COLS - 1) / PR_COLS), 1, q);
    col_reduce_kernel<true><<<grid, 1024, 0, (cudaStream_t)stream>>>(V, ldx, stride, nullptr, 0, os, lat_var, ldm,
                                                                     npad, mt);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}

int plmc_mix_tasks(const double* lat_mean, const double* lat_var, long long ldm, const double* H,
                   const double* var_add, double* mean, double* var, long long mt, int p, int q, int accumulate,
                   void* stream) {
    if (!lat_mean || !H || !mean || mt <= 0 || p <= 0 || q <= 0 || ldm < mt) return PLMC_ERR_BADARG;
    if ((lat_var == nullptr) != (var == nullptr)) return PLMC_ERR_BADARG;
    dim3 grid((unsigned)((mt + MX_J - 1) / MX_J), (p + MX_T - 1) / MX_T);
    mix_tasks_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(lat_mean, lat_var, ldm, H, var_add, mean, var, mt, p, q,
                                                             accumulate);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}
}
