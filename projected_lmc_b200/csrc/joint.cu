// Joint predictive covariance and posterior draws of the task-level posterior.
//
// The eval-mode posterior of ProjectedGPModel (projected_lmc.py:1149-1155) has the covariance
//   T = sum_l C_l (x) h_l h_l^T + I (x) S,     C_l = K**_l - V_l^T V_l,  V_l = L_l^-1 K*_l,
// point-major / task-minor, with S = eps I (+ F F^T after full_likelihood).  The C_l [q, m, m] (lower 128-tiles)
// come from plmc_gram (K**) and plmc_syrk_batched (V^T V) in the factorisation layer; the two kernels here are the
// task-level epilogues:
//   task_covariance  expands the q latent blocks into T, either dense [N, N] or as the lower 128-tiles of an
//                    npad(N)-order matrix with identity padding (the operand of plmc_potrf_batched);
//   mix_samples      maps latent draws G_l = chol(C_l) eps_l and task-level normals E to samples
//                    out[s, j, t] = mean[j, t] + sum_l G[l, j, s] H[l, t] + sum_u E[s, j, u] R[t, u].
// Drawing through the latent structure costs q m^3/3 + q m^2 S; a root of the dense T would cost (n* p)^3 / 3.
#include "plmc_common.cuh"

namespace plmc {

constexpr int TC_THREADS = 256;
constexpr int TC_COLS = 4;   // columns per thread: one CTA writes 1024 consecutive entries of one row of T

// T[a, b] with a = (i, t), b = (j, s): sum_l C_l[max(i,j), min(i,j)] H[l,t] H[l,s] + [i == j] S[t, s].
// Only entries on or below the diagonal of C_l are read.  The product H[l,t] H[l,s] is formed before it
// multiplies C, so T[a, b] and T[b, a] are the same floating-point expression: T is exactly symmetric when S is.
// tiled != 0: only the 128-tiles on or below the diagonal are written, rows / columns >= N are identity padding.
__global__ void __launch_bounds__(TC_THREADS) task_covariance_kernel(
    const double* __restrict__ C, long long ldc, long long stride, const double* __restrict__ H,
    const double* __restrict__ S, double* __restrict__ T, long long ldt, int N, int order, int p, int q, int tiled) {
    const int a = blockIdx.x;
    const int b0 = blockIdx.y * (TC_THREADS * TC_COLS);
    if (tiled && (b0 >> 7) > (a >> 7)) return;
    double* Trow = T + (long long)a * ldt;
    const bool real_row = a < N;
    const int i = real_row ? a / p : 0;
    const int t = real_row ? a - i * p : 0;
#pragma unroll
    for (int c = 0; c < TC_COLS; ++c) {
        const int b = b0 + c * TC_THREADS + threadIdx.x;
        if (b >= order || (tiled && (b >> 7) > (a >> 7))) break;
        double v;
        if (!real_row || b >= N) {
            v = (a == b) ? 1.0 : 0.0;
        } else {
            const int j = b / p;
            const int s = b - j * p;
            const double* Cp = C + (long long)max(i, j) * ldc + min(i, j);
            v = 0.0;
            for (int l = 0; l < q; ++l) v = fma(Cp[(long long)l * stride], H[l * p + t] * H[l * p + s], v);
            if (i == j) v += S[t * p + s];
        }
        Trow[b] = v;
    }
}

constexpr int MS_S = 32;   // samples per CTA (one test point)
constexpr int MS_T = 64;   // tasks per CTA
constexpr int MS_K = 16;   // latents / noise components staged per step

// CTA: one test point j, 32 consecutive samples, 64 tasks; thread = one task x 8 samples.  The samples of a CTA are
// consecutive in G's last dimension (coalesced reads of G without transposing it) and each output row segment
// out[s, j, t0 .. t0+63] is written once.
__global__ void __launch_bounds__(256) mix_samples_kernel(const double* __restrict__ mean, const double* __restrict__ G,
                                                          long long ldg, long long strideg,
                                                          const double* __restrict__ H, const double* __restrict__ E,
                                                          const double* __restrict__ R, double* __restrict__ out,
                                                          long long ns, long long S, int p, int q) {
    __shared__ double Hs[MS_K][MS_T];
    __shared__ double Rs[MS_K][MS_T + 1];
    __shared__ double Gs[MS_K][MS_S];
    __shared__ double Es[MS_S][MS_K + 1];
    const int tid = threadIdx.x;
    const long long nsc = (S + MS_S - 1) / MS_S;
    const long long j = blockIdx.x / nsc;
    const long long s0 = (blockIdx.x - j * nsc) * MS_S;
    const int t0 = blockIdx.y * MS_T;
    const int tl = tid & (MS_T - 1), sg = tid >> 6;   // 4 sample groups x 64 tasks
    double acc[MS_S / 4];
#pragma unroll
    for (int a = 0; a < MS_S / 4; ++a) acc[a] = 0.0;

    // latent part: sum_l G[l, j, s] H[l, t]
    for (int l0 = 0; l0 < q; l0 += MS_K) {
        __syncthreads();
        for (int idx = tid; idx < MS_K * MS_T; idx += 256) {
            const int k = idx / MS_T, tt = idx % MS_T;
            Hs[k][tt] = (l0 + k < q && t0 + tt < p) ? H[(long long)(l0 + k) * p + t0 + tt] : 0.0;
        }
        for (int idx = tid; idx < MS_K * MS_S; idx += 256) {
            const int k = idx / MS_S, ss = idx % MS_S;
            Gs[k][ss] = (l0 + k < q && s0 + ss < S) ? G[(long long)(l0 + k) * strideg + j * ldg + s0 + ss] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < MS_K; ++k) {
            const double h = Hs[k][tl];
#pragma unroll
            for (int a = 0; a < MS_S / 4; ++a) acc[a] = fma(Gs[k][sg + 4 * a], h, acc[a]);
        }
    }
    // task-level noise: sum_u E[s, j, u] R[t, u]
    for (int u0 = 0; u0 < p; u0 += MS_K) {
        __syncthreads();
        for (int idx = tid; idx < MS_K * MS_T; idx += 256) {
            const int k = idx % MS_K, tt = idx / MS_K;
            Rs[k][tt] = (u0 + k < p && t0 + tt < p) ? R[(long long)(t0 + tt) * p + u0 + k] : 0.0;
        }
        for (int idx = tid; idx < MS_S * MS_K; idx += 256) {
            const int k = idx % MS_K, ss = idx / MS_K;
            Es[ss][k] = (u0 + k < p && s0 + ss < S) ? E[((s0 + ss) * ns + j) * p + u0 + k] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < MS_K; ++k) {
            const double r = Rs[k][tl];
#pragma unroll
            for (int a = 0; a < MS_S / 4; ++a) acc[a] = fma(Es[sg + 4 * a][k], r, acc[a]);
        }
    }
    const int t = t0 + tl;
    if (t >= p) return;
    const double mu = mean[j * p + t];
#pragma unroll
    for (int a = 0; a < MS_S / 4; ++a) {
        const long long s = s0 + sg + 4 * a;
        if (s < S) out[(s * ns + j) * p + t] = mu + acc[a];
    }
}

}  // namespace plmc

using namespace plmc;

extern "C" {

int plmc_task_covariance(const double* C, long long ldc, long long stride, const double* H, const double* S,
                         double* T, long long ldt, long long ns, int p, int q, int tiled, void* stream) {
    if (!C || !H || !S || !T || ns <= 0 || p <= 0 || q <= 0 || ldc < ns || (tiled != 0 && tiled != 1))
        return PLMC_ERR_BADARG;
    const long long N = ns * (long long)p;
    const long long order = tiled ? ((N + 127) / 128) * 128 : N;
    const long long col_blocks = (order + TC_THREADS * TC_COLS - 1) / (TC_THREADS * TC_COLS);
    if (order > 2147483647LL || ldt < order || col_blocks > 65535 || stride < 0) return PLMC_ERR_BADARG;
    dim3 grid((unsigned)order, (unsigned)col_blocks);
    task_covariance_kernel<<<grid, TC_THREADS, 0, (cudaStream_t)stream>>>(C, ldc, stride, H, S, T, ldt, (int)N,
                                                                           (int)order, p, q, tiled);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}

int plmc_mix_samples(const double* mean, const double* G, long long ldg, long long strideg, const double* H,
                     const double* E, const double* R, double* out, long long ns, long long S, int p, int q,
                     void* stream) {
    if (!mean || !G || !H || !E || !R || !out || ns <= 0 || S <= 0 || p <= 0 || q <= 0 || ldg < S || strideg < 0)
        return PLMC_ERR_BADARG;
    const long long blocks = ns * ((S + MS_S - 1) / MS_S);
    const long long tblocks = (p + MS_T - 1) / MS_T;
    if (blocks > 2147483647LL || tblocks > 65535) return PLMC_ERR_BADARG;
    dim3 grid((unsigned)blocks, (unsigned)tblocks);
    mix_samples_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(mean, G, ldg, strideg, H, E, R, out, ns, S, p, q);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}
}
