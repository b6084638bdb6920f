// Gradients of the eval-mode predictive means and variances with respect to the test inputs: what autograd gives
// through gpytorch's exact_prediction in the reference (ProjectedGPModel.__call__, projected_lmc.py:1121-1155).
//
// Per latent l and additive component g (z = (x - xbar_g) / ell_{l,g}, s_ij = |z_i - z*_j|^2, K*_l = sum_g o k_g(s)):
//   mu_l(j) = sum_i alpha_l[i] K*_l[i,j],   v_l(j) = k_l(0) - |L_l^-1 K*_l[:,j]|^2.
// With latent cotangents gm_l, gv_l (the transpose of the task mixing, mix_tasks_bwd_kernel) and
// beta_l = K_l^-1 K*_l (two triangular products per test tile, done by the caller only when gv != 0):
//   w[i,j] = gm[j] alpha[i] - 2 gv[j] beta[i,j],   A[i,j] = w[i,j] o k'(s_ij),
//   d/dx*_{jk} += sum_l (2 / ell_{l,k}) (z*_{jk} sum_i A[i,j] - sum_i A[i,j] z_{ik}).
// The prior variance k(x*, x*) is constant for these stationary kernels and contributes nothing.
//
// cross_grad_kernel has the shape of the training sweep's GEMM form (grad_sweep2_kernel, csrc/gram.cu) with the
// roles of the two sides swapped: a CTA owns 64 test points (the row side) and walks a chunk of 128-point train
// tiles (the column side):
//   1. S = Z*_tile Z_tile^T on DMMA -> s = max(|z*|^2 + |z|^2 - 2 S, 0), exactly the forward cross-Gram's s;
//   2. A = w o k'(s) in place (rolled loop; beta is the only O(q n n*) stream and is read once, not at all when
//      there are no variance cotangents);
//   3. U += A Z_tile on DMMA, with the row sums of A taken from the same fragments.
// U and the row sums stay in registers across the chunk, so each test point's gradient is accumulated in a fixed
// order; per-(chunk, latent) partials are reduced by cross_grad_reduce_kernel, which applies 2 / ell per latent
// before the latent sum.  Deterministic, no atomics.  Inputs of up to 48 padded dimensions take the same kernel with
// zero-padded DMMA operands (dpad <= 24: two CTAs per SM).
#include "kernel_math.cuh"
#include "plmc_b200.h"

namespace plmc {

constexpr int CG_THREADS = 256;
constexpr int CG_ROWS = 64;        // test points per CTA
constexpr int CG_AS = 132;         // row stride of At: = 4 mod 16, conflict-free DMMA A-fragment loads
constexpr int CG_TARGET_CTAS = 592;
constexpr int CG_MAX_DPAD = 48;

__host__ __device__ inline int cg_lds(int nb) { return nb * 8 + 4; }   // = 4 mod 8; columns [dpad, lds) are zero
__host__ __device__ inline size_t cg_smem(int nb) {
    return (size_t)((128 + CG_ROWS) * cg_lds(nb) + CG_ROWS * CG_AS + 128 + 2 * CG_ROWS) * 8;
}
static inline int cg_nb(int dpad) { return dpad <= 8 ? 1 : (dpad <= 16 ? 2 : (dpad <= 24 ? 3 : 6)); }

static inline int cg_chunks(long long npad, long long ns, int q) {
    const long long row_tiles = npad / 128;
    const long long base = ((ns + CG_ROWS - 1) / CG_ROWS) * q;
    long long c = (CG_TARGET_CTAS + base - 1) / base;
    if (c > row_tiles) c = row_tiles;
    if (c < 1) c = 1;
    const long long per = (row_tiles + c - 1) / c;     // no empty chunk
    return (int)((row_tiles + per - 1) / per);
}

// A = w o k'(s) over this thread's entries of At (s parked there by step 1; a thread reads back only its own slots)
template <int KID>
__device__ __forceinline__ void cg_transform(double* __restrict__ At, const double* __restrict__ aj,
                                             const double* __restrict__ gms, const double* __restrict__ gvs,
                                             const double* __restrict__ bl, long long ldb, long long t0,
                                             long long i0, long long n, long long ns, int wm, int wn, int g, int t,
                                             double osl, KernelShape sh) {
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        const int cl = wn * 32 + j * 8 + 2 * t;
        const double2 ajv = *reinterpret_cast<const double2*>(aj + cl);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = wm * 32 + i * 8 + g;
            const bool row_ok = t0 + rl < ns;
            const double gm = gms[rl], gv2 = -2.0 * gvs[rl];
            double2* slot = reinterpret_cast<double2*>(At + rl * CG_AS + cl);
            const double2 sv = *slot;
            double out[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const long long gi = i0 + cl + e;
                double w = 0.0;
                if (row_ok && gi < n) {
                    w = gm * (e ? ajv.y : ajv.x);
                    if (bl) w = fma(gv2, __ldg(bl + gi * ldb + t0 + rl), w);
                }
                double kk, dk, dka;
                kernel_value_grad<KID>(e ? sv.y : sv.x, kk, dk, dka, sh);
                out[e] = w * (osl * dk);
            }
            *slot = make_double2(out[0], out[1]);
        }
    }
}

template <int KID, int NB>
__global__ void __launch_bounds__(CG_THREADS, (NB <= 3 ? 2 : 1))
    cross_grad_kernel(const double* __restrict__ Ztr, const double* __restrict__ zntr, long long npad,
                      const double* __restrict__ Zte, const double* __restrict__ znte, long long rows_pad_te,
                      const double* __restrict__ alpha, long long lda, const double* __restrict__ g_mean,
                      const double* __restrict__ g_var, long long ldg, const double* __restrict__ beta, long long ldb,
                      long long strideb, const double* __restrict__ os, const double* __restrict__ shape,
                      double* __restrict__ partial, long long rows_part, long long n, long long ns, int dpad,
                      int tiles_per_chunk) {
    extern __shared__ __align__(16) double sm[];
    constexpr int lds = NB * 8 + 4;
    double* Zj = sm;                       // [128][lds]  train tile
    double* Zi = Zj + 128 * lds;           // [64][lds]   test points of this CTA
    double* At = Zi + CG_ROWS * lds;       // [64][CG_AS]
    double* aj = At + CG_ROWS * CG_AS;     // [128]
    double* gms = aj + 128;                // [64]
    double* gvs = gms + CG_ROWS;           // [64]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    const int l = blockIdx.z, ch = blockIdx.y, q = gridDim.z;
    const long long t0 = (long long)blockIdx.x * CG_ROWS;
    const double osl = os ? os[l] : 1.0;
    const KernelShape sh = (KID == 4) ? kernel_shape(shape[l]) : KernelShape{0.0, 0.0};
    const double* Zl = Ztr + (long long)l * npad * dpad;
    const double* znl = zntr + (long long)l * npad;
    const double* al = alpha + (long long)l * lda;
    const double* bl = beta ? beta + (long long)l * strideb : nullptr;
    const int dp2 = dpad >> 1;
    const long long row_tiles = npad / 128;
    const long long tb = (long long)ch * tiles_per_chunk;
    const long long te = min(row_tiles, tb + tiles_per_chunk);

    for (int idx = tid; idx < 192 * (lds - dpad); idx += CG_THREADS) {
        const int r = idx / (lds - dpad), c = idx - r * (lds - dpad);
        Zj[r * lds + dpad + c] = 0.0;      // Zi follows Zj with the same row stride: rows 128..191 are Zi
    }
    {
        const int rr = tid >> 2;
        const double2* src = reinterpret_cast<const double2*>(Zte + ((long long)l * rows_pad_te + t0 + rr) * dpad);
        double2* dst = reinterpret_cast<double2*>(Zi + rr * lds);
        for (int c = tid & 3; c < dp2; c += 4) dst[c] = __ldg(src + c);
    }
    if (tid < CG_ROWS) {
        const bool ok = t0 + tid < ns;
        gms[tid] = (ok && g_mean) ? g_mean[(long long)l * ldg + t0 + tid] : 0.0;
        gvs[tid] = (ok && g_var) ? g_var[(long long)l * ldg + t0 + tid] : 0.0;
    }
    double ni[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) ni[i] = __ldg(znte + (long long)l * rows_pad_te + t0 + wm * 32 + i * 8 + g);

    double u[NB][2];
#pragma unroll
    for (int nb = 0; nb < NB; ++nb) u[nb][0] = u[nb][1] = 0.0;
    double ra = 0.0;

    for (long long tile = tb; tile < te; ++tile) {
        const long long i0 = tile * 128;
        __syncthreads();                   // the previous tile's readers of Zj / aj / At are done
        {
            const int rr = tid >> 1;
            const double2* src = reinterpret_cast<const double2*>(Zl + (i0 + rr) * dpad);
            double2* dst = reinterpret_cast<double2*>(Zj + rr * lds);
            for (int c = tid & 1; c < dp2; c += 2) dst[c] = __ldg(src + c);
            if (tid < 128) aj[tid] = (i0 + tid < n) ? al[i0 + tid] : 0.0;
        }
        double nj[4][2];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double2 v = __ldg(reinterpret_cast<const double2*>(znl + i0 + wn * 32 + j * 8 + 2 * t));
            nj[j][0] = v.x;
            nj[j][1] = v.y;
        }
        __syncthreads();                   // Zj / aj (and, on the first tile, Zi / gms / gvs) staged

        // ---- 1. cross term on DMMA, squared distances into At
        {
            double acc[4][4][2];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
            const double* pa = Zi + (wm * 32 + g) * lds + t;
            const double* pb = Zj + (wn * 32 + g) * lds + t;
            for (int k0 = 0; k0 < dpad; k0 += 4) {
                double af[4], bf[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) af[i] = pa[i * 8 * lds + k0];
#pragma unroll
                for (int j = 0; j < 4; ++j) bf[j] = pb[j * 8 * lds + k0];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const double s0 = dmax(fma(-2.0, acc[i][j][0], ni[i] + nj[j][0]), 0.0);
                    const double s1 = dmax(fma(-2.0, acc[i][j][1], ni[i] + nj[j][1]), 0.0);
                    *reinterpret_cast<double2*>(At + (wm * 32 + i * 8 + g) * CG_AS + wn * 32 + j * 8 + 2 * t) =
                        make_double2(s0, s1);
                }
        }
        // ---- 2. A = w o k'(s) in place
        cg_transform<KID>(At, aj, gms, gvs, bl, ldb, t0, i0, n, ns, wm, wn, g, t, osl, sh);
        __syncthreads();                   // At = A complete

        // ---- 3. U += A Z_tile on DMMA (warp w: test rows 8w..8w+7), row sums of A from the same fragments
        {
            const double* pa = At + (warp * 8 + g) * CG_AS + t;
            const double* pb = Zj + t * lds + g;
#pragma unroll 4
            for (int kk = 0; kk < 32; ++kk) {
                const double a = pa[kk * 4];
                ra += a;
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) dmma884(u[nb][0], u[nb][1], a, pb[kk * 4 * lds + nb * 8]);
            }
        }
    }
    ra += __shfl_xor_sync(0xffffffffu, ra, 1);
    ra += __shfl_xor_sync(0xffffffffu, ra, 2);

    // sum_i A_ij (z*_jk - z_ik) = z*_jk ra_j - U_jk for test row warp*8+g, dimensions nb*8 + 2t + e
    const int row = warp * 8 + g;
    const double* pz = Zi + row * lds + 2 * t;
    double* pp = partial + (((long long)ch * q + l) * rows_part + t0 + row) * dpad;
#pragma unroll
    for (int nb = 0; nb < NB; ++nb)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int k = nb * 8 + 2 * t + e;
            if (k < dpad) pp[k] = fma(pz[nb * 8 + e], ra, -u[nb][e]);
        }
}

// g_x[j, k] = sum_l (2 / ell[l, k]) sum_c partial[c, l, j, k]   (fixed order: chunks, then latents)
__global__ void cross_grad_reduce_kernel(const double* __restrict__ partial, const double* __restrict__ ell,
                                         double* __restrict__ g_x, long long ldx, long long rows_part, long long ns,
                                         int d, int dpad, int q, int chunks) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ns * d) return;
    const long long j = idx / d;
    const int k = (int)(idx - j * d);
    double s = 0.0;
    for (int l = 0; l < q; ++l) {
        double c = 0.0;
        for (int ch = 0; ch < chunks; ++ch) c += partial[(((long long)ch * q + l) * rows_part + j) * dpad + k];
        s = fma(2.0 / ell[(long long)l * d + k], c, s);
    }
    g_x[j * ldx + k] = s;
}

// The transpose of mix_tasks_kernel: gm_l[j] = sum_t g_mean[j,t] H[l,t],  gv_l[j] = sum_t g_var[j,t] H[l,t]^2
__global__ void __launch_bounds__(256) mix_tasks_bwd_kernel(const double* __restrict__ g_mean,
                                                            const double* __restrict__ g_var,
                                                            const double* __restrict__ H, double* __restrict__ g_lm,
                                                            double* __restrict__ g_lv, long long ldm, long long mt,
                                                            int p) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int l = blockIdx.y;
    if (j >= mt) return;
    const double* h = H + (long long)l * p;
    double sm_ = 0.0, sv = 0.0;
    for (int t = 0; t < p; ++t) {
        const double ht = h[t];
        if (g_mean) sm_ = fma(g_mean[j * p + t], ht, sm_);
        if (g_var) sv = fma(g_var[j * p + t], ht * ht, sv);
    }
    if (g_lm) g_lm[(long long)l * ldm + j] = sm_;
    if (g_lv) g_lv[(long long)l * ldm + j] = sv;
}

}  // namespace plmc

using namespace plmc;

extern "C" {

long long plmc_cross_grad_ws(long long npad, long long ns, int d, int q) {
    if (npad <= 0 || (npad % 128) || ns <= 0 || d <= 0 || q <= 0) return 0;
    const int dpad = ((d + 3) / 4) * 4;
    const long long rows_part = ((ns + CG_ROWS - 1) / CG_ROWS) * CG_ROWS;
    return 8LL * cg_chunks(npad, ns, q) * q * rows_part * dpad;
}

int plmc_cross_grad(const double* Ztrain, const double* zntrain, long long npad, const double* Ztest,
                    const double* zntest, long long rows_pad_test, int kernel_id, const double* os,
                    const double* shape, const double* ell, const double* alpha, long long lda, const double* g_mean,
                    const double* g_var, long long ldg, const double* beta, long long ldb, long long strideb,
                    double* g_x, long long ldx, double* partial, long long n, long long ns, int d, int dpad, int q,
                    void* stream) {
    const long long rows_part = ((ns + CG_ROWS - 1) / CG_ROWS) * CG_ROWS;
    if (!Ztrain || !zntrain || !Ztest || !zntest || !ell || !alpha || !g_x || !partial || n <= 0 || npad < n ||
        (npad % 128) || ns <= 0 || rows_pad_test < rows_part || d <= 0 || dpad != ((d + 3) / 4) * 4 ||
        dpad > CG_MAX_DPAD || q <= 0 || q > 65535 || lda < n || ldx < d || kernel_id < 0 ||
        kernel_id > PLMC_KERNEL_RQ || (kernel_id == PLMC_KERNEL_RQ) != (shape != nullptr) ||
        (!g_mean && !g_var) || ldg < ns || (g_var == nullptr) != (beta == nullptr) ||
        (beta && (ldb < ns || strideb < npad * ldb)))
        return PLMC_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int chunks = cg_chunks(npad, ns, q);
    const long long row_tiles = npad / 128;
    const int per = (int)((row_tiles + chunks - 1) / chunks);
    const int nb = cg_nb(dpad);
    const size_t smem = cg_smem(nb);
    dim3 grid((unsigned)(rows_part / CG_ROWS), chunks, q);
#define PLMC_CG_LAUNCH(KID, NB)                                                                                     \
    {                                                                                                               \
        cudaFuncSetAttribute(cross_grad_kernel<KID, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
        cross_grad_kernel<KID, NB><<<grid, CG_THREADS, smem, st>>>(Ztrain, zntrain, npad, Ztest, zntest,           \
                                                                   rows_pad_test, alpha, lda, g_mean, g_var, ldg,  \
                                                                   beta, ldb, strideb, os, shape, partial,         \
                                                                   rows_part, n, ns, dpad, per);                   \
    }
#define PLMC_CG_CASE(KID)                              \
    case KID:                                          \
        if (nb == 1) PLMC_CG_LAUNCH(KID, 1)            \
        else if (nb == 2) PLMC_CG_LAUNCH(KID, 2)       \
        else if (nb == 3) PLMC_CG_LAUNCH(KID, 3)       \
        else PLMC_CG_LAUNCH(KID, 6)                    \
        break;
    switch (kernel_id) {
        PLMC_CG_CASE(0)
        PLMC_CG_CASE(1)
        PLMC_CG_CASE(2)
        PLMC_CG_CASE(3)
        PLMC_CG_CASE(4)
        default: return PLMC_ERR_BADARG;
    }
#undef PLMC_CG_CASE
#undef PLMC_CG_LAUNCH
    PLMC_CHECK_LAUNCH();
    const long long work = ns * d;
    cross_grad_reduce_kernel<<<(unsigned)((work + 255) / 256), 256, 0, st>>>(partial, ell, g_x, ldx, rows_part, ns, d,
                                                                            dpad, q, chunks);
    PLMC_CHECK_LAUNCH();
    note_launch(2);
    return PLMC_OK;
}

int plmc_mix_tasks_bwd(const double* g_mean, const double* g_var, const double* H, double* g_lat_mean,
                       double* g_lat_var, long long ldm, long long mt, int p, int q, void* stream) {
    if (!H || mt <= 0 || p <= 0 || q <= 0 || q > 65535 || ldm < mt || (!g_mean && !g_var) ||
        (g_mean == nullptr) != (g_lat_mean == nullptr) || (g_var == nullptr) != (g_lat_var == nullptr))
        return PLMC_ERR_BADARG;
    dim3 grid((unsigned)((mt + 255) / 256), q);
    mix_tasks_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g_mean, g_var, H, g_lat_mean, g_lat_var, ldm, mt, p);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}
}
