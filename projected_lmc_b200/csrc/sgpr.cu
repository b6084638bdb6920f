// Adjoint of the cross-Gram block K[l, i, j] = os[l] k(|zr_i - zc_j|^2): the piece of autograd the
// inducing-point (SGPR, Titsias 2009) variant of the model needs (ExactGPModel(..., n_inducing_points=m),
// projected_lmc.py:302-303 -> gpytorch InducingPointKernel).  Given the cotangent G = dL/dK [q, nr, nc] it returns
//   g_ell[l, k]  = dL/d ell[l, k]    = sum_ij G_ij os dk/ds (-2 (zr_ik - zc_jk)^2 / ell_lk)
//   g_os[l]      = dL/d os[l]        = sum_ij G_ij k(s_ij)
//   g_shape[l]   = dL/d alpha[l]     = sum_ij G_ij os dk/dalpha     (RQ only; slot dpad + 1 of part_ell)
//   g_rows[i, k] = dL/d (row point i, dimension k), summed over the latents (the inducing points are shared):
//                  sum_l sum_j G_ij os dk/ds 2 (zr_ik - zc_jk) / ell_lk
// without materialising dK/dtheta.  Rows are the m inducing points (a few hundred), columns the n training or test
// points: one CTA owns 128 rows and walks a chunk of the columns, so every row gradient is accumulated by ONE
// thread in a fixed order (deterministic; no atomics); per-chunk partials are reduced by a second tiny kernel.
// The n x m work is ~100 flop per pair -- milliseconds at SARCOS size; the m x m and n x m algebra around it
// (Cholesky of K_uu, two triangular solves, one Gram product) is plain library work done in torch.
#include "kernel_math.cuh"
#include "plmc_b200.h"

namespace plmc {

constexpr int SG_DC = 16;        // dimensions accumulated per pass (registers: 2 x 16 doubles per thread)
constexpr int SG_COLS = 128;     // columns per tile
constexpr int SG_THREADS = 256;  // 128 rows x 2 column halves

template <int KID>
__global__ void __launch_bounds__(SG_THREADS, 1)
    cross_gram_bwd_kernel(const double* __restrict__ Zr, long long rows_pad_r, const double* __restrict__ Zc,
                          long long rows_pad_c, const double* __restrict__ G, long long ldg, long long strideG,
                          const double* __restrict__ os, const double* __restrict__ ell, double* __restrict__ part_rows,
                          double* __restrict__ part_ell, long long nr, long long nc, int d, int dpad, int chunks,
                          long long cols_per_chunk, const double* __restrict__ shape) {
    extern __shared__ __align__(16) double sm[];
    const int ldz = dpad + 1;
    double* Zrs = sm;                          // [128][ldz]
    double* Zcs = Zrs + 128 * ldz;             // [128][ldz]
    double* Gs = Zcs + 128 * ldz;              // [128][129]
    double* red = Gs + 128 * 129;              // [8][SG_DC + 1]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = tid & 127, half = tid >> 7;
    const int rt = blockIdx.x, ch = blockIdx.y, l = blockIdx.z;
    const int q = gridDim.z, row_tiles = gridDim.x;
    const long long i0 = (long long)rt * 128;
    const double osl = os ? os[l] : 1.0;
    const KernelShape sh = (KID == 4) ? kernel_shape(shape[l]) : KernelShape{0.0, 0.0};
    const int nslot = dpad + 1 + (KID == 4 ? 1 : 0);   // part_ell slots per (chunk, latent, row tile)
    const double* zr = Zr + ((long long)l * rows_pad_r + i0) * dpad;
    const double* zc = Zc + (long long)l * rows_pad_c * dpad;
    const double* Gl = G + (long long)l * strideG;
    const long long j_beg = (long long)ch * cols_per_chunk;
    const long long j_end = min(nc, j_beg + cols_per_chunk);

    for (int idx = tid; idx < 128 * dpad; idx += SG_THREADS) {
        const int r = idx / dpad, k = idx - r * dpad;
        Zrs[r * ldz + k] = (i0 + r < rows_pad_r) ? zr[idx] : 0.0;
    }
    const int npass = (dpad + SG_DC - 1) / SG_DC;
    for (int pass = 0; pass < npass; ++pass) {
        const int k0 = pass * SG_DC;
        const int kc = min(SG_DC, dpad - k0);
        double au[SG_DC], al[SG_DC];
#pragma unroll
        for (int k = 0; k < SG_DC; ++k) au[k] = al[k] = 0.0;
        double a_os = 0.0, a_al = 0.0;
        for (long long j0 = j_beg; j0 < j_end; j0 += SG_COLS) {
            __syncthreads();
            for (int idx = tid; idx < 128 * dpad; idx += SG_THREADS) {
                const int r = idx / dpad, k = idx - r * dpad;
                Zcs[r * ldz + k] = (j0 + r < rows_pad_c) ? zc[(j0 + r) * dpad + k] : 0.0;
            }
            for (int idx = tid; idx < 128 * SG_COLS; idx += SG_THREADS) {
                const int r = idx >> 7, c = idx & 127;
                Gs[r * 129 + c] = (i0 + r < nr && j0 + c < j_end) ? Gl[(i0 + r) * ldg + j0 + c] : 0.0;
            }
            __syncthreads();
            const double* zi = Zrs + row * ldz;
            for (int c = half * 64; c < half * 64 + 64; ++c) {
                const double g = Gs[row * 129 + c];
                const double* zj = Zcs + c * ldz;
                double s = 0.0;
                for (int k = 0; k < dpad; ++k) {
                    const double dlt = zi[k] - zj[k];
                    s = fma(dlt, dlt, s);
                }
                double kk, dk, dka;
                kernel_value_grad<KID>(s, kk, dk, dka, sh);
                if (pass == 0) a_os = fma(g, kk, a_os);
                if (KID == 4 && pass == 0) a_al = fma(g, dka, a_al);
                const double w = g * osl * dk;
#pragma unroll
                for (int k = 0; k < SG_DC; ++k) {
                    if (k < kc) {
                        const double dlt = zi[k0 + k] - zj[k0 + k];
                        au[k] = fma(w, dlt, au[k]);
                        al[k] = fma(w * dlt, dlt, al[k]);
                    }
                }
            }
        }
        // row gradients: one slot per (chunk, half, latent, row); factor 2 / ell_lk applied here so the sum over
        // latents in the reduction is a plain sum
        double* pr = part_rows + ((((long long)ch * 2 + half) * q + l) * row_tiles * 128 + i0 + row) * dpad + k0;
#pragma unroll
        for (int k = 0; k < SG_DC; ++k)
            if (k < kc) pr[k] = (k0 + k < d) ? 2.0 * au[k] / ell[(long long)l * d + k0 + k] : 0.0;
        // lengthscale / outputscale partials of this CTA: fixed-order reduction over its 256 threads
        // (slot k < SG_DC: sum_ij w_ij dz_k^2 ; slot SG_DC: sum_ij G_ij k(s_ij), slot SG_DC + 1 (RQ):
        // sum_ij G_ij os dk/dalpha, first pass only)
#pragma unroll
        for (int k = 0; k <= SG_DC + (KID == 4 ? 1 : 0); ++k) {
            const bool is_os = (k == SG_DC), is_al = (k == SG_DC + 1);
            if ((is_os || is_al) ? (pass != 0) : (k >= kc)) continue;      // uniform over the CTA
            double v = warp_sum(is_al ? osl * a_al : (is_os ? a_os : al[k < SG_DC ? k : 0]));
            __syncthreads();
            if (lane == 0) red[warp] = v;
            __syncthreads();
            if (tid == 0) {
                double t = 0.0;
                for (int w8 = 0; w8 < SG_THREADS / 32; ++w8) t += red[w8];
                double* pe = part_ell + (((long long)ch * q + l) * row_tiles + rt) * nslot;
                pe[is_al ? dpad + 1 : (is_os ? dpad : k0 + k)] = t;
            }
        }
    }
}

// g_rows[i, k] = sum over (chunk, half, latent) partial ; g_ell[l, k] = -(2/ell) sum over (chunk, row tile) ; g_os
__global__ void cross_gram_bwd_reduce_kernel(const double* __restrict__ part_rows, const double* __restrict__ part_ell,
                                             const double* __restrict__ ell, double* __restrict__ g_rows,
                                             double* __restrict__ g_ell, double* __restrict__ g_os, long long nr, int d,
                                             int dpad, int q, int chunks, int row_tiles, int has_shape,
                                             double* __restrict__ g_shape) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long rows_all = (long long)row_tiles * 128;
    if (t < nr * d) {
        const long long i = t / d;
        const int k = (int)(t - i * d);
        double s = 0.0;
        for (int c = 0; c < chunks * 2; ++c)
            for (int l = 0; l < q; ++l) s += part_rows[(((long long)c * q + l) * rows_all + i) * dpad + k];
        g_rows[t] = s;
    }
    const int per = d + 1 + has_shape, nslot = dpad + 1 + has_shape;
    if (t < (long long)q * per) {
        const int l = (int)(t / per), k = (int)(t - (long long)l * per);
        double s = 0.0;
        for (int c = 0; c < chunks; ++c)
            for (int r = 0; r < row_tiles; ++r)
                s += part_ell[(((long long)c * q + l) * row_tiles + r) * nslot + (k < d ? k : dpad + (k - d))];
        if (k < d) g_ell[(long long)l * d + k] = -2.0 * s / ell[(long long)l * d + k];
        else if (k == d) {
            if (g_os) g_os[l] = s;
        } else if (g_shape)
            g_shape[l] = s;
    }
}

static inline int sgpr_chunks(long long nc) {
    long long c = (nc + 4095) / 4096;
    return (int)(c < 1 ? 1 : (c > 64 ? 64 : c));
}

}  // namespace plmc

using namespace plmc;

extern "C" {

long long plmc_cross_gram_bwd_ws(long long nr, long long nc, int d, int q) {
    return plmc_cross_gram_bwd_ws2(nr, nc, d, q, PLMC_KERNEL_RBF);
}

long long plmc_cross_gram_bwd_ws2(long long nr, long long nc, int d, int q, int kernel_id) {
    if (nr <= 0 || nc <= 0 || d <= 0 || q <= 0) return 0;
    const int dpad = ((d + 3) / 4) * 4;
    const int nslot = dpad + 1 + (kernel_id == PLMC_KERNEL_RQ ? 1 : 0);
    const long long row_tiles = (nr + 127) / 128;
    const int chunks = sgpr_chunks(nc);
    return 8LL * ((long long)chunks * 2 * q * row_tiles * 128 * dpad + (long long)chunks * q * row_tiles * nslot);
}

int plmc_cross_gram_bwd(const double* Zr, long long rows_pad_r, const double* Zc, long long rows_pad_c, const double* G,
                        long long ldg, long long strideG, int kernel_id, const double* os, const double* ell,
                        double* g_ell, double* g_os, double* g_rows, double* partial, long long nr, long long nc, int d,
                        int dpad, int q, void* stream) {
    return plmc_cross_gram_bwd2(Zr, rows_pad_r, Zc, rows_pad_c, G, ldg, strideG, kernel_id, os, nullptr, ell, g_ell,
                                g_os, nullptr, g_rows, partial, nr, nc, d, dpad, q, stream);
}

int plmc_cross_gram_bwd2(const double* Zr, long long rows_pad_r, const double* Zc, long long rows_pad_c,
                         const double* G, long long ldg, long long strideG, int kernel_id, const double* os,
                         const double* shape, const double* ell, double* g_ell, double* g_os, double* g_shape,
                         double* g_rows, double* partial, long long nr, long long nc, int d, int dpad, int q,
                         void* stream) {
    if (!Zr || !Zc || !G || !ell || !g_ell || !g_rows || !partial || nr <= 0 || nc <= 0 || d <= 0 || dpad < d ||
        (dpad & 3) || q <= 0 || q > 65535 || ldg < nc || rows_pad_r < nr || rows_pad_c < nc ||
        (kernel_id == PLMC_KERNEL_RQ) != (shape != nullptr) || (g_shape && !shape))
        return PLMC_ERR_BADARG;
    const int has_shape = shape != nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    const int row_tiles = (int)((nr + 127) / 128);
    const int chunks = sgpr_chunks(nc);
    long long cols = (nc + chunks - 1) / chunks;
    cols = ((cols + SG_COLS - 1) / SG_COLS) * SG_COLS;
    double* part_rows = partial;
    double* part_ell = partial + (long long)chunks * 2 * q * row_tiles * 128 * dpad;
    const size_t smem = (size_t)(2 * 128 * (dpad + 1) + 128 * 129 + 16) * 8;
    if (smem > 227 * 1024) return PLMC_ERR_BADARG;
    dim3 grid(row_tiles, chunks, q);
#define PLMC_SGPR_CASE(KID)                                                                                          \
    case KID:                                                                                                        \
        cudaFuncSetAttribute(cross_gram_bwd_kernel<KID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);    \
        cross_gram_bwd_kernel<KID><<<grid, SG_THREADS, smem, st>>>(Zr, rows_pad_r, Zc, rows_pad_c, G, ldg, strideG, os, \
                                                                   ell, part_rows, part_ell, nr, nc, d, dpad, chunks, \
                                                                   cols, shape);                                      \
        break;
    switch (kernel_id) {
        PLMC_SGPR_CASE(0)
        PLMC_SGPR_CASE(1)
        PLMC_SGPR_CASE(2)
        PLMC_SGPR_CASE(3)
        PLMC_SGPR_CASE(4)
        default: return PLMC_ERR_BADARG;
    }
#undef PLMC_SGPR_CASE
    PLMC_CHECK_LAUNCH();
    const long long per = (long long)q * (d + 1 + has_shape);
    const long long work = (nr * d > per) ? nr * d : per;
    cross_gram_bwd_reduce_kernel<<<(unsigned)((work + 255) / 256), 256, 0, st>>>(part_rows, part_ell, ell, g_rows, g_ell,
                                                                                g_os, nr, d, dpad, q, chunks, row_tiles,
                                                                                has_shape, g_shape);
    PLMC_CHECK_LAUNCH();
    note_launch(2);
    return PLMC_OK;
}
}
