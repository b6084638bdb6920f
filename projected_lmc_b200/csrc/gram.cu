// Kernel (2): batched ARD Gram construction (training K + sigma^2 I and the
// train x test cross block), and kernel (4): the fused backward sweep.
//
// Gram semantics follow gpytorch 1.11 as reached from handle_covar_
// (projected_lmc.py:151-167, evaluated by log_prob at :1201):
//   x -> (x - mean_rows(x)) / lengthscale,  s_ij = |zi|^2 + |zj|^2 - 2 zi.zj,
//   clamp_min(0); RBF exp(-s/2); Matern: r = sqrt(max(s, 1e-30)),
//   nu=5/2: (1 + sqrt5 r + 5/3 r^2) exp(-sqrt5 r); ScaleKernel multiplies by
//   the outputscale; GaussianLikelihood adds sigma^2 on the diagonal (:1200).
// The cross term zi.zj runs on the FP64 tensor cores (DMMA.8x8x4), the
// transform, outputscale, noise/jitter and the identity padding are fused into
// the epilogue: K is written exactly once (lower 128-tiles only).
//
// Algorithmic bytes: 8*q*n(n+1)/2 written (Gram), the same read (sweep).
#include "kernel_math.cuh"
#include "plmc_b200.h"

namespace plmc {

constexpr int GR_THREADS = 256;
constexpr int GR_KC = 32;  // input-dimension chunk staged in shared memory by the Gram kernel


// xmean[k] = mean_i X[i, k]
__global__ void __launch_bounds__(256) col_mean_kernel(const double* __restrict__ X, long long n, int d,
                                                       double* __restrict__ xmean) {
    __shared__ double sh[32];
    const int k = blockIdx.x;
    double s = 0.0;
    for (long long i = threadIdx.x; i < n; i += 256) s += X[i * d + k];
    s = block_sum<256>(s, sh);
    if (threadIdx.x == 0) xmean[k] = s / (double)n;
}

__global__ void __launch_bounds__(256) scale_inputs_kernel(const double* __restrict__ X,
                                                           const double* __restrict__ xmean,
                                                           const double* __restrict__ ell, double* __restrict__ Z,
                                                           double* __restrict__ zn, long long n, int d, int dpad,
                                                           long long rows_pad) {
    const int l = blockIdx.z;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows_pad) return;
    double* z = Z + ((long long)l * rows_pad + i) * dpad;
    double s = 0.0;
    for (int k = 0; k < dpad; ++k) {
        double v = 0.0;
        if (i < n && k < d) v = (X[i * d + k] - xmean[k]) / ell[(long long)l * d + k];
        z[k] = v;
        s = fma(v, v, s);
    }
    zn[(long long)l * rows_pad + i] = s;
}

// MODE 0: training Gram (lower tiles, diagonal noise, identity padding)
// MODE 1: cross Gram (all tiles; rows >= n are zero)
// A 128 x 128 tile is processed as two 64-row halves by 8 warps (2 x 4, 32 x 32 entries each): 64 accumulator
// registers per thread and a 64 KB staging slab, so that TWO CTAs fit an SM for d <= 24 (109 KB, <= 128 registers)
// and the load / DMMA phase of one overlaps the transcendental phase of the other (ncu of the one-CTA version: FP64
// pipe 26 % active, 8 warps per SM, top stall "wait").  Wider inputs are staged in chunks of GR_KC dimensions.
__host__ __device__ inline int gram_kc(int dpad) { return dpad <= 24 ? dpad : GR_KC; }
__host__ __device__ inline int gram_lds(int kc) { return (kc % 8 == 0) ? kc + 4 : kc + 8; }   // = 4 mod 8
__host__ __device__ inline size_t gram_smem(int dpad) {
    return (size_t)(192 * gram_lds(gram_kc(dpad)) + 32 * GR_THREADS) * 8;
}

template <int KID, int MODE>
__global__ void __launch_bounds__(GR_THREADS, 2)
    gram_kernel(const double* __restrict__ Zr, const double* __restrict__ znr, long long rows_pad_r,
                const double* __restrict__ Zc, const double* __restrict__ znc, long long rows_pad_c,
                const double* __restrict__ os, const double* __restrict__ diag_add, double* __restrict__ Kout,
                long long ld, long long stride, long long n, int dpad, int tiles_c, int accumulate,
                const double* __restrict__ shape) {
    extern __shared__ __align__(16) double sm[];
    const int kcmax = gram_kc(dpad);
    const int lds = gram_lds(kcmax);
    double* Zj = sm;                     // [128][lds]
    double* Zi = Zj + 128 * lds;         // [64][lds]
    double* stage = Zi + 64 * lds;       // [32][256]: slot e of thread tid at stage[e * 256 + tid]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    const int l = blockIdx.z;

    int ti, tj;
    if (MODE == 0) {
        const long long b = blockIdx.x;
        int r = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
        while ((long long)(r + 1) * (r + 2) / 2 <= b) ++r;
        while ((long long)r * (r + 1) / 2 > b) --r;
        ti = r;
        tj = (int)(b - (long long)r * (r + 1) / 2);
    } else {
        ti = blockIdx.x / tiles_c;
        tj = blockIdx.x - ti * tiles_c;
    }
    const long long i0 = (long long)ti * 128, j0 = (long long)tj * 128;
    const double* zc = Zc + ((long long)l * rows_pad_c + j0) * dpad;
    const double osl = os ? os[l] : 1.0;
    const KernelShape sh = (KID == 4) ? kernel_shape(shape[l]) : KernelShape{0.0, 0.0};
    const double dadd = (MODE == 0) ? diag_add[l] : 0.0;
    double* Kl = Kout + (long long)l * stride;
    const bool single = dpad <= kcmax;   // one chunk: the column side is staged once per tile

    double nj[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const double2 v =
            __ldg(reinterpret_cast<const double2*>(znc + (long long)l * rows_pad_c + j0 + wn * 32 + j * 8 + 2 * t));
        nj[j][0] = v.x;
        nj[j][1] = v.y;
    }

    for (int h = 0; h < 2; ++h) {
        const long long ih0 = i0 + 64 * h;
        const double* zr = Zr + ((long long)l * rows_pad_r + ih0) * dpad;
        double ni[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) ni[i] = __ldg(znr + (long long)l * rows_pad_r + ih0 + wm * 32 + i * 8 + g);

        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        const double* pa = Zi + (wm * 32 + g) * lds + t;
        const double* pb = Zj + (wn * 32 + g) * lds + t;
        for (int kc0 = 0; kc0 < dpad; kc0 += kcmax) {
            const int kc = min(kcmax, dpad - kc0);
            const int kc2 = kc >> 1;
            __syncthreads();             // previous readers of Zi (and Zj when it is restaged) are done
            {
                const int rr = tid >> 2;
                const double2* src = reinterpret_cast<const double2*>(zr + rr * dpad + kc0);
                double2* dst = reinterpret_cast<double2*>(Zi + rr * lds);
                for (int c = tid & 3; c < kc2; c += 4) dst[c] = __ldg(src + c);
            }
            if (!single || h == 0) {
                const int rr = tid >> 1;
                const double2* src = reinterpret_cast<const double2*>(zc + rr * dpad + kc0);
                double2* dst = reinterpret_cast<double2*>(Zj + rr * lds);
                for (int c = tid & 1; c < kc2; c += 2) dst[c] = __ldg(src + c);
            }
            __syncthreads();
            for (int k0 = 0; k0 < kc; k0 += 4) {
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
        }

        // Squared distances into the thread's private slots (conflict free; a thread reads back only what it
        // wrote, so no barrier), then the transcendental epilogue as a ROLLED loop: fully unrolled it is tens of KB
        // of code and the kernel stalls on instruction fetch.
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                stage[((i * 4 + j) * 2 + 0) * GR_THREADS + tid] = dmax(fma(-2.0, acc[i][j][0], ni[i] + nj[j][0]), 0.0);
                stage[((i * 4 + j) * 2 + 1) * GR_THREADS + tid] = dmax(fma(-2.0, acc[i][j][1], ni[i] + nj[j][1]), 0.0);
            }
        // Interior half tiles (99 % of them at n = 44k: off the diagonal, no padded row or column) take a loop
        // without any per-element predicate; diagonal and edge tiles the general one.
        const bool interior = (MODE == 0) ? (ti != tj && i0 + 128 <= n) : (ih0 + 64 <= n);
        if (interior) {
            double* base = Kl + (ih0 + wm * 32 + g) * ld + j0 + wn * 32 + 2 * t;
#pragma unroll 4
            for (int pr = 0; pr < 16; ++pr) {
                const int i = pr >> 2, j = pr & 3;
                double* dst = base + (long long)(i * 8) * ld + j * 8;
                double v0 = osl * kernel_value<KID>(stage[(pr * 2 + 0) * GR_THREADS + tid], sh);
                double v1 = osl * kernel_value<KID>(stage[(pr * 2 + 1) * GR_THREADS + tid], sh);
                if (accumulate) {
                    const double2 old = *reinterpret_cast<const double2*>(dst);
                    v0 += old.x;
                    v1 += old.y;
                }
                *reinterpret_cast<double2*>(dst) = make_double2(v0, v1);
            }
            continue;
        }
#pragma unroll 4
        for (int pr = 0; pr < 16; ++pr) {
            const int i = pr >> 2, j = pr & 3;
            const long long gi = ih0 + wm * 32 + i * 8 + g;
            const long long gj = j0 + wn * 32 + j * 8 + 2 * t;
            double v[2];
            // accumulate: a further component of an additive kernel (sum_g os_g k_g) is added onto the tile; the
            // noise diagonal and the identity padding were written with the first component
            double2 old = make_double2(0.0, 0.0);
            if (accumulate) old = *reinterpret_cast<const double2*>(Kl + gi * ld + gj);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const long long gje = gj + e;
                double s = stage[(pr * 2 + e) * GR_THREADS + tid];
                if (MODE == 0) {
                    if (gi == gje) s = 0.0;
                    double kv = osl * kernel_value<KID>(s, sh);
                    if (gi == gje && !accumulate) kv += dadd;
                    if (gi >= n || gje >= n) kv = (gi == gje && !accumulate) ? 1.0 : 0.0;
                    v[e] = kv;
                } else {
                    v[e] = (gi < n) ? osl * kernel_value<KID>(s, sh) : 0.0;
                }
            }
            *reinterpret_cast<double2*>(Kl + gi * ld + gj) = make_double2(v[0] + old.x, v[1] + old.y);
        }
    }
}

// ---------------------------------------------------------------------------
// Fused backward sweep.  With W = 1/2 (alpha alpha^T - K^-1) and the symmetric
// weights w_ij (2 below the diagonal, 1 on it), one pass over the lower tiles of
// K^-1 accumulates, per latent:
//   acc[k]      = sum w_ij W_ij os dk/ds (z_ik - z_jk)^2      k < d
//   acc[dpad]   = sum w_ij W_ij k(s_ij)                        (d lp / d os)
//   acc[dpad+1] = sum_i W_ii                                   (d lp / d sigma^2)
// K tiles are recomputed from Z (direct differences); dK is never materialised.
// partial layout: [q, gridDim.x, dpad + 2]; the reduction is fixed-order.
// ---------------------------------------------------------------------------
template <int KID>
__global__ void __launch_bounds__(GR_THREADS, 1)
    grad_sweep_kernel(const double* __restrict__ Kinv, long long ld, long long stride,
                      const double* __restrict__ alpha, long long lda_vec, const double* __restrict__ Z,
                      const double* __restrict__ os, double* __restrict__ partial, long long n, long long npad,
                      int dpad, long long ntiles, const double* __restrict__ shape) {
    extern __shared__ __align__(16) double sm[];
    const int lds = dpad + 1;
    double* Zi = sm;                    // [128][lds]
    double* Zj = Zi + 128 * lds;        // [128][lds]
    double* ai = Zj + 128 * lds;        // [128]
    double* aj = ai + 128;              // [128]
    double* wsum = aj + 128;            // [8][nacc]
    double* cta_acc = wsum + 8 * (dpad + 2 + (KID == 4 ? 1 : 0));  // [nacc]
    double* stage = cta_acc + (dpad + 2 + (KID == 4 ? 1 : 0));     // [64][256] private per-thread slots

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    const int l = blockIdx.z;
    const int nacc = dpad + 2 + (KID == 4 ? 1 : 0);   // + sum w W dk/dalpha (RQ)
    const double osl = os ? os[l] : 1.0;
    const KernelShape sh = (KID == 4) ? kernel_shape(shape[l]) : KernelShape{0.0, 0.0};
    const double* Kl = Kinv + (long long)l * stride;
    const double* al = alpha + (long long)l * lda_vec;
    const double* Zl = Z + (long long)l * npad * dpad;

    if (tid < nacc) cta_acc[tid] = 0.0;

    for (long long b = blockIdx.x; b < ntiles; b += gridDim.x) {
        int r = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
        while ((long long)(r + 1) * (r + 2) / 2 <= b) ++r;
        while ((long long)r * (r + 1) / 2 > b) --r;
        const int ti = r, tj = (int)(b - (long long)r * (r + 1) / 2);
        const long long i0 = (long long)ti * 128, j0 = (long long)tj * 128;

        __syncthreads();
        for (int idx = tid; idx < 128 * dpad; idx += GR_THREADS) {
            const int rr = idx / dpad, k = idx - rr * dpad;
            Zi[rr * lds + k] = Zl[i0 * dpad + idx];
            Zj[rr * lds + k] = Zl[j0 * dpad + idx];
        }
        if (tid < 128) {
            ai[tid] = (i0 + tid < n) ? al[i0 + tid] : 0.0;
            aj[tid] = (j0 + tid < n) ? al[j0 + tid] : 0.0;
        }
        __syncthreads();

        // thread patch: rows wm*64 + 8*i + g (i<8), cols wn*32 + 8*j + 2t + e (j<4, e<2)
        double Wv[8][8];  // first s_ij, then A_ij = w * W * os * dk/ds
        const int rbase = wm * 64 + g, cbase = wn * 32 + 2 * t;
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int c = 0; c < 8; ++c) Wv[i][c] = 0.0;
        // squared scaled distances by direct differences
        for (int k = 0; k < dpad; ++k) {
            double zi[8], zj[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) zi[i] = Zi[(rbase + i * 8) * lds + k];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                zj[2 * j] = Zj[(cbase + j * 8) * lds + k];
                zj[2 * j + 1] = Zj[(cbase + j * 8 + 1) * lds + k];
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const double dlt = zi[i] - zj[c];
                    Wv[i][c] = fma(dlt, dlt, Wv[i][c]);
                }
        }
        // The transcendental transform runs as a ROLLED loop over this thread's 32 element pairs
        // (values parked in a private shared-memory slab, slot e at stage[e*256+tid]; no barrier:
        // a thread only reads back what it wrote).  Fully unrolled it overflows the instruction cache.
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int c = 0; c < 8; ++c) stage[(i * 8 + c) * GR_THREADS + tid] = Wv[i][c];
        double s_os = 0.0, s_tr = 0.0, s_al = 0.0;
#pragma unroll 4
        for (int pr = 0; pr < 32; ++pr) {
            const int i = pr >> 2, j = pr & 3;
            const long long gi = i0 + rbase + i * 8;
            const double a_i = ai[rbase + i * 8];
            const int cl0 = cbase + j * 8;
            const double2 kv = *reinterpret_cast<const double2*>(Kl + gi * ld + j0 + cl0);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int cl = cl0 + e;
                const long long gj = j0 + cl;
                double w = (gj < gi) ? 2.0 : (gj == gi ? 1.0 : 0.0);
                if (gi >= n || gj >= n) w = 0.0;
                const double Wij = (w != 0.0) ? 0.5 * (a_i * aj[cl] - (e ? kv.y : kv.x)) : 0.0;
                double kk, dk, dka;
                kernel_value_grad<KID>(stage[(pr * 2 + e) * GR_THREADS + tid], kk, dk, dka, sh);
                s_os = fma(w * Wij, kk, s_os);
                if (KID == 4) s_al = fma(w * Wij, dka, s_al);
                if (gj == gi && gi < n) s_tr += Wij;
                stage[(pr * 2 + e) * GR_THREADS + tid] = w * Wij * osl * dk;
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int c = 0; c < 8; ++c) Wv[i][c] = stage[(i * 8 + c) * GR_THREADS + tid];
        // per-dimension accumulation  sum A_ij (z_ik - z_jk)^2
        for (int k = 0; k < dpad; ++k) {
            double zi[8], zj[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) zi[i] = Zi[(rbase + i * 8) * lds + k];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                zj[2 * j] = Zj[(cbase + j * 8) * lds + k];
                zj[2 * j + 1] = Zj[(cbase + j * 8 + 1) * lds + k];
            }
            double sk = 0.0;
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const double dlt = zi[i] - zj[c];
                    sk = fma(Wv[i][c], dlt * dlt, sk);
                }
            sk = warp_sum(sk);
            if (lane == 0) wsum[warp * nacc + k] = sk;
        }
        s_os = warp_sum(s_os);
        s_tr = warp_sum(s_tr);
        if (KID == 4) s_al = warp_sum(s_al);
        if (lane == 0) {
            wsum[warp * nacc + dpad] = s_os;
            wsum[warp * nacc + dpad + 1] = s_tr;
            if (KID == 4) wsum[warp * nacc + dpad + 2] = s_al;
        }
        __syncthreads();
        if (tid < nacc) {
            double s = 0.0;
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) s += wsum[w8 * nacc + tid];
            cta_acc[tid] += s;
        }
    }
    __syncthreads();
    if (tid < nacc) partial[((long long)l * gridDim.x + blockIdx.x) * nacc + tid] = cta_acc[tid];
}

// ---------------------------------------------------------------------------
// Fused backward sweep, GEMM form (input dimension d <= 24; the kernel above remains for wider inputs).
// Both contractions of the sweep run on the FP64 tensor cores and the CTA is small enough for two per SM, so the
// load / DMMA phases of one overlap the transcendental phase of the other:
//   1. cross term  S = Zi Zj^T (DMMA)  ->  s_ij = max(|zi|^2 + |zj|^2 - 2 S_ij, 0), exactly the forward Gram's s;
//   2. transform (rolled loop over the thread's entries, parked in the tile buffer At):
//        A_ij = w_ij W_ij os dk/ds(s_ij)   (0 on the diagonal),   s_os += w W k,   s_tr += W_ii;
//   3. sum_ij A_ij (z_ik - z_jk)^2 = sum_i z_ik (ra_i z_ik - 2 U_ik) + sum_j ca_j z_jk^2   with U = A Zj (DMMA,
//      64 x 128 x d), ra / ca the row / column sums of A (ra falls out of the A fragments the DMMA loads anyway).
// A 128 x 128 tile of the lower triangle is processed as two 64-row halves.  Shared memory (d <= 24): Zj 128 x 28,
// Zi 64 x 28, At 64 x 132 doubles + 3 KB = 111 KB, registers <= 128: two CTAs per SM.
// Per-thread partial sums live in registers across the CTA's whole tile sequence; one fixed-order reduction at
// the end (deterministic).  partial layout as above: [q, gridDim.x, dpad + 2].
// ---------------------------------------------------------------------------
constexpr int SW_AS = 132;   // row stride of At: = 4 mod 16, conflict-free DMMA A-fragment loads
__host__ __device__ inline int sweep_lds(int dpad) { return (dpad % 8 == 0) ? dpad + 4 : dpad + 8; }
__host__ __device__ inline size_t sweep2_smem(int dpad) {
    return (size_t)((128 + 64) * sweep_lds(dpad) + 64 * SW_AS + 128 + 256) * 8;
}

template <int KID, bool INTERIOR>
__device__ __forceinline__ void sweep_transform(double* __restrict__ At, const double* __restrict__ aj,
                                                const double* __restrict__ Kl, long long ld, long long ih0,
                                                long long j0, long long n, int wm, int wn, int g, int t,
                                                const double (&ai)[4], double osl, double& s_os, double& s_tr,
                                                KernelShape sh, double& s_al) {
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        const int cl = wn * 32 + j * 8 + 2 * t;
        const long long gj = j0 + cl;
        const double2 ajv = *reinterpret_cast<const double2*>(aj + cl);
        double2 kv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            kv[i] = __ldg(reinterpret_cast<const double2*>(Kl + (ih0 + wm * 32 + i * 8 + g) * ld + gj));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = wm * 32 + i * 8 + g;
            const long long gi = ih0 + rl;
            double2* slot = reinterpret_cast<double2*>(At + rl * SW_AS + cl);
            const double2 sv = *slot;
            double out[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const double raw = fma(ai[i], e ? ajv.y : ajv.x, -(e ? kv[i].y : kv[i].x));   // 2 W_ij
                double kk, dk, dka;
                kernel_value_grad<KID>(e ? sv.y : sv.x, kk, dk, dka, sh);
                if (INTERIOR) {                       // strictly below the diagonal, no padding: w/2 = 1
                    s_os = fma(raw, kk, s_os);
                    if (KID == 4) s_al = fma(raw, dka, s_al);
                    out[e] = raw * (osl * dk);
                } else {
                    const long long gje = gj + e;
                    double w = (gje < gi) ? 1.0 : ((gje == gi) ? 0.5 : 0.0);
                    if (gi >= n || gje >= n) w = 0.0;
                    const double c1 = (w != 0.0) ? w * raw : 0.0;   // entries above the diagonal are never used
                    s_os = fma(c1, kk, s_os);
                    if (KID == 4) s_al = fma(c1, dka, s_al);
                    if (gje == gi) s_tr += c1;
                    out[e] = (gje == gi) ? 0.0 : c1 * (osl * dk);
                }
            }
            *slot = make_double2(out[0], out[1]);
        }
    }
}

template <int KID, int NB>
__global__ void __launch_bounds__(GR_THREADS, 2)
    grad_sweep2_kernel(const double* __restrict__ Kinv, long long ld, long long stride,
                       const double* __restrict__ alpha, long long lda_vec, const double* __restrict__ Z,
                       const double* __restrict__ zn, const double* __restrict__ os, double* __restrict__ partial,
                       long long n, long long npad, int dpad, long long ntiles, const double* __restrict__ shape) {
    extern __shared__ __align__(16) double sm[];
    const int lds = sweep_lds(dpad);
    double* Zj = sm;                     // [128][lds]
    double* Zi = Zj + 128 * lds;         // [64][lds]
    double* At = Zi + 64 * lds;          // [64][SW_AS]
    double* aj = At + 64 * SW_AS;        // [128]
    double* ca2 = aj + 128;              // [2][128]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp >> 2, wn = warp & 3;
    const int l = blockIdx.z;
    const int nacc = dpad + 2 + (KID == 4 ? 1 : 0);
    const double osl = os ? os[l] : 1.0;
    const KernelShape sh = (KID == 4) ? kernel_shape(shape[l]) : KernelShape{0.0, 0.0};
    const double* Kl = Kinv + (long long)l * stride;
    const double* al = alpha + (long long)l * lda_vec;
    const double* Zl = Z + (long long)l * npad * dpad;
    const double* znl = zn + (long long)l * npad;
    const int dp2 = dpad >> 1;           // double2 per row of Z

    // the padding columns [dpad, lds) of the staged inputs are read by the last 8-wide dimension block: zero, once
    for (int idx = tid; idx < 192 * (lds - dpad); idx += GR_THREADS) {
        const int r = idx / (lds - dpad), c = idx - r * (lds - dpad);
        Zj[r * lds + dpad + c] = 0.0;    // Zi follows Zj with the same row stride: rows 128..191 are Zi
    }

    double gacc[NB][2];                  // dims nb*8 + 2t + e, summed over this thread's rows (all tiles)
#pragma unroll
    for (int nb = 0; nb < NB; ++nb) gacc[nb][0] = gacc[nb][1] = 0.0;
    double cacc = 0.0;                   // dim = lane, column-side term
    double s_os = 0.0, s_tr = 0.0, s_al = 0.0;   // s_al: sum w W dk/dalpha (RQ only)

    for (long long b = blockIdx.x; b < ntiles; b += gridDim.x) {
        int r = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
        while ((long long)(r + 1) * (r + 2) / 2 <= b) ++r;
        while ((long long)r * (r + 1) / 2 > b) --r;
        const int ti = r, tj = (int)(b - (long long)r * (r + 1) / 2);
        const long long i0 = (long long)ti * 128, j0 = (long long)tj * 128;
        const bool interior = (ti != tj) && (i0 + 128 <= n);

        __syncthreads();                 // everyone is done with Zj / aj / ca2 of the previous tile
        {
            const int rr = tid >> 1;
            const double2* src = reinterpret_cast<const double2*>(Zl + (j0 + rr) * dpad);
            double2* dst = reinterpret_cast<double2*>(Zj + rr * lds);
            for (int c = tid & 1; c < dp2; c += 2) dst[c] = __ldg(src + c);
            if (tid < 128) aj[tid] = (j0 + tid < n) ? al[j0 + tid] : 0.0;
        }
        double nj[4][2];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double2 v = __ldg(reinterpret_cast<const double2*>(znl + j0 + wn * 32 + j * 8 + 2 * t));
            nj[j][0] = v.x;
            nj[j][1] = v.y;
        }

        for (int h = 0; h < 2; ++h) {
            const long long ih0 = i0 + 64 * h;
            {
                const int rr = tid >> 2;
                const double2* src = reinterpret_cast<const double2*>(Zl + (ih0 + rr) * dpad);
                double2* dst = reinterpret_cast<double2*>(Zi + rr * lds);
                for (int c = tid & 3; c < dp2; c += 4) dst[c] = __ldg(src + c);
            }
            double ai[4], ni[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const long long gi = ih0 + wm * 32 + i * 8 + g;
                ai[i] = (gi < n) ? __ldg(al + gi) : 0.0;
                ni[i] = __ldg(znl + gi);
            }
            __syncthreads();             // Zi (and, for h = 0, Zj / aj) staged

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
                        *reinterpret_cast<double2*>(At + (wm * 32 + i * 8 + g) * SW_AS + wn * 32 + j * 8 + 2 * t) =
                            make_double2(s0, s1);
                    }
            }
            // ---- 2. transform in place (a thread reads back only the slots it wrote: no barrier)
            if (interior)
                sweep_transform<KID, true>(At, aj, Kl, ld, ih0, j0, n, wm, wn, g, t, ai, osl, s_os, s_tr, sh, s_al);
            else
                sweep_transform<KID, false>(At, aj, Kl, ld, ih0, j0, n, wm, wn, g, t, ai, osl, s_os, s_tr, sh, s_al);
            __syncthreads();             // At = A complete

            // ---- 3. U = A Zj on DMMA (warp w: rows 8w..8w+7), row sums from the same fragments, column sums
            {
                double u[NB][2];
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) u[nb][0] = u[nb][1] = 0.0;
                double ra = 0.0;
                const double* pa = At + (warp * 8 + g) * SW_AS + t;
                const double* pb = Zj + t * lds + g;
#pragma unroll 4
                for (int kk = 0; kk < 32; ++kk) {
                    const double a = pa[kk * 4];
                    ra += a;
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) dmma884(u[nb][0], u[nb][1], a, pb[kk * 4 * lds + nb * 8]);
                }
                ra += __shfl_xor_sync(0xffffffffu, ra, 1);
                ra += __shfl_xor_sync(0xffffffffu, ra, 2);
                {
                    const int col = tid & 127, hf = tid >> 7;
                    const double* pc = At + (hf * 32) * SW_AS + col;
                    double c = 0.0;
#pragma unroll 8
                    for (int rr = 0; rr < 32; ++rr) c += pc[rr * SW_AS];
                    ca2[hf * 128 + col] = c;
                }
                const double* pz = Zi + (warp * 8 + g) * lds + 2 * t;
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) {
                    const double2 z = *reinterpret_cast<const double2*>(pz + nb * 8);
                    gacc[nb][0] = fma(z.x, fma(ra, z.x, -2.0 * u[nb][0]), gacc[nb][0]);
                    gacc[nb][1] = fma(z.y, fma(ra, z.y, -2.0 * u[nb][1]), gacc[nb][1]);
                }
            }
            __syncthreads();             // ca2 visible; At / Zi free for the next half
            if (lane < NB * 8) {
#pragma unroll 4
                for (int m = 0; m < 16; ++m) {
                    const int jj = warp + 8 * m;
                    const double zz = Zj[jj * lds + lane];
                    cacc = fma((ca2[jj] + ca2[128 + jj]) * zz, zz, cacc);
                }
            }
        }
    }

    // ---- fixed-order reduction of the per-thread sums: over the row lanes g, then over the 8 warps
    __syncthreads();
    double* red = At;                    // [8][nacc] (+ [8][NB*8] for the column-side sums)
    double* red2 = At + 8 * nacc;
#pragma unroll
    for (int nb = 0; nb < NB; ++nb)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            double v = gacc[nb][e];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            const int k = nb * 8 + 2 * t + e;
            if (g == 0 && k < dpad) red[warp * nacc + k] = v;
        }
    if (lane < NB * 8) red2[warp * (NB * 8) + lane] = cacc;
    s_os = warp_sum(s_os);
    s_tr = warp_sum(s_tr);
    if (KID == 4) s_al = warp_sum(s_al);
    if (lane == 0) {
        red[warp * nacc + dpad] = s_os;
        red[warp * nacc + dpad + 1] = s_tr;
        if (KID == 4) red[warp * nacc + dpad + 2] = s_al;
    }
    __syncthreads();
    if (tid < nacc) {
        double s = 0.0;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) s += red[w8 * nacc + tid];
        if (tid < dpad) {
            double c = 0.0;
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) c += red2[w8 * (NB * 8) + tid];
            s += c;
        }
        partial[((long long)l * gridDim.x + blockIdx.x) * nacc + tid] = s;
    }
}

// g_ell[l,k] = -(2/ell[l,k]) * sum_c partial[l,c,k] ; g_os, g_noise likewise; with a shape parameter (nacc =
// dpad + 3) g_shape[l] = os[l] * sum_c partial[l,c,dpad+2]
__global__ void grad_reduce_kernel(const double* __restrict__ partial, int chunks, int d, int dpad,
                                   const double* __restrict__ ell, double* __restrict__ g_ell,
                                   double* __restrict__ g_os, double* __restrict__ g_noise, int nacc,
                                   const double* __restrict__ os, double* __restrict__ g_shape) {
    const int l = blockIdx.x;
    for (int a = threadIdx.x; a < nacc; a += blockDim.x) {
        double s = 0.0;
        for (int c = 0; c < chunks; ++c) s += partial[((long long)l * chunks + c) * nacc + a];
        if (a < d)
            g_ell[(long long)l * d + a] = -2.0 * s / ell[(long long)l * d + a];
        else if (a == dpad) {
            if (g_os) g_os[l] = s;
        } else if (a == dpad + 1)
            g_noise[l] = s;
        else if (a == dpad + 2 && g_shape)
            g_shape[l] = (os ? os[l] : 1.0) * s;
    }
}

static inline int sweep_ctas(long long ntiles) { return (int)(ntiles < 592 ? ntiles : 592); }

// the shape argument of the ...2 entry points: required by RQ, refused by the kernels without a shape parameter
static inline bool shape_arg_ok(int kernel_id, const double* shape) {
    return (kernel_id == PLMC_KERNEL_RQ) == (shape != nullptr);
}

}  // namespace plmc

using namespace plmc;

// diagnostics (tests): force the direct-difference sweep kernel for every input dimension
static bool g_sweep_direct = false;

template <int MODE>
static int launch_gram(int kernel_id, dim3 grid, size_t smem, cudaStream_t st, const double* Zr, const double* znr,
                       long long rpr, const double* Zc, const double* znc, long long rpc, const double* os,
                       const double* diag_add, double* K, long long ld, long long stride, long long n, int dpad,
                       int tiles_c, int accumulate, const double* shape) {
#define PLMC_GRAM_CASE(KID)                                                                                     \
    case KID:                                                                                                   \
        if (smem > 48 * 1024)                                                                                   \
            cudaFuncSetAttribute(gram_kernel<KID, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        gram_kernel<KID, MODE><<<grid, GR_THREADS, smem, st>>>(Zr, znr, rpr, Zc, znc, rpc, os, diag_add, K, ld,  \
                                                               stride, n, dpad, tiles_c, accumulate, shape);    \
        break;
    switch (kernel_id) {
        PLMC_GRAM_CASE(0)
        PLMC_GRAM_CASE(1)
        PLMC_GRAM_CASE(2)
        PLMC_GRAM_CASE(3)
        PLMC_GRAM_CASE(4)
        default: return PLMC_ERR_BADARG;
    }
#undef PLMC_GRAM_CASE
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}

extern "C" {

/* host only (no device work): k(s) and dk/ds of kernel `kernel_id` evaluated with the SAME source the device
 * kernels compile (csrc/kernel_math.cuh) -- lets the CPU test-suite check the hand-written exp / sqrt. */
int plmc_kernel_profile_host(int kernel_id, const double* s_host, long long n, double* k_host, double* dk_host) {
    if (!s_host || !k_host || !dk_host || n < 0) return PLMC_ERR_BADARG;
    for (long long i = 0; i < n; ++i) {
        switch (kernel_id) {
            case 0: kernel_value_grad<0>(s_host[i], k_host[i], dk_host[i]); break;
            case 1: kernel_value_grad<1>(s_host[i], k_host[i], dk_host[i]); break;
            case 2: kernel_value_grad<2>(s_host[i], k_host[i], dk_host[i]); break;
            case 3: kernel_value_grad<3>(s_host[i], k_host[i], dk_host[i]); break;
            default: return PLMC_ERR_BADARG;
        }
    }
    return PLMC_OK;
}

/* host only: k(s), dk/ds and dk/dshape with the device source, shape[i] the kernel's shape parameter for s[i]
 * (RQ: alpha; NULL for kernels 0-3, whose dk/dshape is 0) */
int plmc_kernel_profile2_host(int kernel_id, const double* s_host, const double* shape_host, long long n,
                              double* k_host, double* dk_host, double* dshape_host) {
    if (!s_host || !k_host || !dk_host || !dshape_host || n < 0 || kernel_id < 0 || kernel_id > PLMC_KERNEL_RQ ||
        !shape_arg_ok(kernel_id, shape_host))
        return PLMC_ERR_BADARG;
    for (long long i = 0; i < n; ++i) {
        switch (kernel_id) {
            case 0: kernel_value_grad<0>(s_host[i], k_host[i], dk_host[i], dshape_host[i], KernelShape{}); break;
            case 1: kernel_value_grad<1>(s_host[i], k_host[i], dk_host[i], dshape_host[i], KernelShape{}); break;
            case 2: kernel_value_grad<2>(s_host[i], k_host[i], dk_host[i], dshape_host[i], KernelShape{}); break;
            case 3: kernel_value_grad<3>(s_host[i], k_host[i], dk_host[i], dshape_host[i], KernelShape{}); break;
            default:
                kernel_value_grad<4>(s_host[i], k_host[i], dk_host[i], dshape_host[i], kernel_shape(shape_host[i]));
        }
    }
    return PLMC_OK;
}

/* host only: log1p(x), x >= 0, as the RQ kernel evaluates it on the device (csrc/kernel_math.cuh) */
int plmc_log1p_host(const double* x_host, long long n, double* out_host) {
    if (!x_host || !out_host || n < 0) return PLMC_ERR_BADARG;
    for (long long i = 0; i < n; ++i) out_host[i] = log1p_nonneg(x_host[i]);
    return PLMC_OK;
}

/* host only: the pivot step of the Cholesky leaf (csrc/kernel_math.cuh sqrt_and_reciprocal) on host arrays */
int plmc_sqrt_reciprocal_host(const double* s_host, long long n, double* root_host, double* inv_host) {
    if (!s_host || !root_host || !inv_host || n < 0) return PLMC_ERR_BADARG;
    for (long long i = 0; i < n; ++i) sqrt_and_reciprocal(s_host[i], root_host[i], inv_host[i]);
    return PLMC_OK;
}

int plmc_col_mean(const double* X, long long n, int d, double* xmean, void* stream) {
    if (!X || !xmean || n <= 0 || d <= 0) return PLMC_ERR_BADARG;
    col_mean_kernel<<<d, 256, 0, (cudaStream_t)stream>>>(X, n, d, xmean);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}

int plmc_scale_inputs(const double* X, const double* xmean, const double* ell, double* Z, double* zn, long long n,
                      int d, int dpad, long long rows_pad, int q, void* stream) {
    if (!X || !xmean || !ell || !Z || !zn || n <= 0 || d <= 0 || dpad < d || (dpad & 3) || rows_pad < n || q <= 0)
        return PLMC_ERR_BADARG;
    dim3 grid((unsigned)((rows_pad + 255) / 256), 1, q);
    scale_inputs_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(X, xmean, ell, Z, zn, n, d, dpad, rows_pad);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}

int plmc_gram(const double* Z, const double* zn, int kernel_id, const double* os, const double* diag_add, double* K,
              long long ld, long long stride, long long n, long long npad, int dpad, int q, int accumulate,
              void* stream) {
    return plmc_gram2(Z, zn, kernel_id, os, nullptr, diag_add, K, ld, stride, n, npad, dpad, q, accumulate, stream);
}

int plmc_gram2(const double* Z, const double* zn, int kernel_id, const double* os, const double* shape,
               const double* diag_add, double* K, long long ld, long long stride, long long n, long long npad, int dpad,
               int q, int accumulate, void* stream) {
    if (!Z || !zn || !diag_add || !K || n <= 0 || npad < n || (npad % 128) || ld < npad || (ld & 1) || dpad <= 0 ||
        (dpad & 3) || q <= 0 || q > 65535 || !shape_arg_ok(kernel_id, shape))
        return PLMC_ERR_BADARG;
    const long long tm = npad / 128;
    const long long tiles = tm * (tm + 1) / 2;
    if (tiles > 2147483647LL) return PLMC_ERR_BADARG;
    const size_t smem = gram_smem(dpad);
    return launch_gram<0>(kernel_id, dim3((unsigned)tiles, 1, q), smem, (cudaStream_t)stream, Z, zn, npad, Z, zn, npad,
                          os, diag_add, K, ld, stride, n, dpad, (int)tm, accumulate, shape);
}

int plmc_cross_gram(const double* Ztrain, const double* zntrain, const double* Ztest, const double* zntest,
                    int kernel_id, const double* os, double* Kx, long long ldx, long long stride, long long n,
                    long long npad, long long mt_rows_pad, long long mt, int dpad, int q, int accumulate,
                    void* stream) {
    return plmc_cross_gram2(Ztrain, zntrain, Ztest, zntest, kernel_id, os, nullptr, Kx, ldx, stride, n, npad,
                            mt_rows_pad, mt, dpad, q, accumulate, stream);
}

int plmc_cross_gram2(const double* Ztrain, const double* zntrain, const double* Ztest, const double* zntest,
                     int kernel_id, const double* os, const double* shape, double* Kx, long long ldx, long long stride,
                     long long n, long long npad, long long mt_rows_pad, long long mt, int dpad, int q, int accumulate,
                     void* stream) {
    if (!Ztrain || !zntrain || !Ztest || !zntest || !Kx || n <= 0 || npad < n || (npad % 128) || mt <= 0 ||
        (mt % 128) || mt_rows_pad < mt || ldx < mt || (ldx & 1) || dpad <= 0 || (dpad & 3) || q <= 0 || q > 65535 ||
        !shape_arg_ok(kernel_id, shape))
        return PLMC_ERR_BADARG;
    const long long tr = npad / 128, tc = mt / 128;
    if (tr * tc > 2147483647LL) return PLMC_ERR_BADARG;
    const size_t smem = gram_smem(dpad);
    return launch_gram<1>(kernel_id, dim3((unsigned)(tr * tc), 1, q), smem, (cudaStream_t)stream, Ztrain, zntrain,
                          npad, Ztest, zntest, mt_rows_pad, os, nullptr, Kx, ldx, stride, n, dpad, (int)tc, accumulate,
                          shape);
}

int plmc_sweep_debug(int direct) {
    g_sweep_direct = direct != 0;
    return PLMC_OK;
}

long long plmc_grad_ws(long long npad, int d, int q) { return plmc_grad_ws2(npad, d, q, PLMC_KERNEL_RBF); }

long long plmc_grad_ws2(long long npad, int d, int q, int kernel_id) {
    if (npad <= 0 || d <= 0 || q <= 0) return 0;
    const long long tm = npad / 128;
    const int dpad = ((d + 3) / 4) * 4;
    const int nacc = dpad + 2 + (kernel_id == PLMC_KERNEL_RQ ? 1 : 0);
    return (long long)q * sweep_ctas(tm * (tm + 1) / 2) * nacc * 8;
}

int plmc_grad_sweep(const double* Kinv, long long ld, long long stride, const double* alpha, long long lda_vec,
                    const double* Z, const double* zn, const double* ell, int kernel_id, const double* os,
                    double* g_ell, double* g_os, double* g_noise, double* partial, long long n, long long npad, int d,
                    int dpad, int q, void* stream) {
    return plmc_grad_sweep2(Kinv, ld, stride, alpha, lda_vec, Z, zn, ell, kernel_id, os, nullptr, g_ell, g_os, g_noise,
                            nullptr, partial, n, npad, d, dpad, q, stream);
}

int plmc_grad_sweep2(const double* Kinv, long long ld, long long stride, const double* alpha, long long lda_vec,
                     const double* Z, const double* zn, const double* ell, int kernel_id, const double* os,
                     const double* shape, double* g_ell, double* g_os, double* g_noise, double* g_shape,
                     double* partial, long long n, long long npad, int d, int dpad, int q, void* stream) {
    if (!Kinv || !alpha || !Z || !zn || !ell || !g_ell || !g_noise || !partial || n <= 0 || npad < n || (npad % 128) ||
        ld < npad || (ld & 1) || d <= 0 || dpad < d || (dpad & 3) || dpad != ((d + 3) / 4) * 4 || q <= 0 ||
        q > 65535 || lda_vec < n || !shape_arg_ok(kernel_id, shape) || (g_shape && !shape))
        return PLMC_ERR_BADARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int nacc = dpad + 2 + (kernel_id == PLMC_KERNEL_RQ ? 1 : 0);
    const long long tm = npad / 128;
    const long long ntiles = tm * (tm + 1) / 2;
    const int ctas = sweep_ctas(ntiles);
    if (dpad <= 24 && !g_sweep_direct) {
        // GEMM form on the FP64 tensor cores, two CTAs per SM
        const size_t smem2 = sweep2_smem(dpad);
        dim3 grid2(ctas, 1, q);
#define PLMC_SWEEP2_LAUNCH(KID, NB)                                                                                \
    {                                                                                                              \
        cudaFuncSetAttribute(grad_sweep2_kernel<KID, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2); \
        grad_sweep2_kernel<KID, NB><<<grid2, GR_THREADS, smem2, st>>>(Kinv, ld, stride, alpha, lda_vec, Z, zn, os,   \
                                                                     partial, n, npad, dpad, ntiles, shape);       \
    }
#define PLMC_SWEEP2_CASE(KID)                                   \
    case KID:                                                   \
        if (dpad <= 8) PLMC_SWEEP2_LAUNCH(KID, 1)               \
        else if (dpad <= 16) PLMC_SWEEP2_LAUNCH(KID, 2)         \
        else PLMC_SWEEP2_LAUNCH(KID, 3)                         \
        break;
        switch (kernel_id) {
            PLMC_SWEEP2_CASE(0)
            PLMC_SWEEP2_CASE(1)
            PLMC_SWEEP2_CASE(2)
            PLMC_SWEEP2_CASE(3)
            PLMC_SWEEP2_CASE(4)
            default: return PLMC_ERR_BADARG;
        }
#undef PLMC_SWEEP2_CASE
#undef PLMC_SWEEP2_LAUNCH
        PLMC_CHECK_LAUNCH();
        note_launch(1);
        grad_reduce_kernel<<<q, 64, 0, st>>>(partial, ctas, d, dpad, ell, g_ell, g_os, g_noise, nacc, os, g_shape);
        PLMC_CHECK_LAUNCH();
        note_launch(1);
        return PLMC_OK;
    }
    const size_t smem = (size_t)(2 * 128 * (dpad + 1) + 256 + 9 * nacc + 64 * GR_THREADS) * 8;
    if (smem > 227 * 1024) return PLMC_ERR_BADARG;
    dim3 grid(ctas, 1, q);
#define PLMC_SWEEP_CASE(KID)                                                                                     \
    case KID:                                                                                                    \
        if (smem > 48 * 1024)                                                                                    \
            cudaFuncSetAttribute(grad_sweep_kernel<KID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        grad_sweep_kernel<KID><<<grid, GR_THREADS, smem, st>>>(Kinv, ld, stride, alpha, lda_vec, Z, os, partial, n, \
                                                               npad, dpad, ntiles, shape);                       \
        break;
    switch (kernel_id) {
        PLMC_SWEEP_CASE(0)
        PLMC_SWEEP_CASE(1)
        PLMC_SWEEP_CASE(2)
        PLMC_SWEEP_CASE(3)
        PLMC_SWEEP_CASE(4)
        default: return PLMC_ERR_BADARG;
    }
#undef PLMC_SWEEP_CASE
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    grad_reduce_kernel<<<q, 64, 0, st>>>(partial, ctas, d, dpad, ell, g_ell, g_os, g_noise, nacc, os, g_shape);
    PLMC_CHECK_LAUNCH();
    note_launch(1);
    return PLMC_OK;
}
}
