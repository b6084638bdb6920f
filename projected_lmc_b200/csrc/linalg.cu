#include "linalg.cuh"
#include "potrf_leaf.cuh"

#include <array>
#include <cstdio>
#include <map>
#include <vector>

namespace plmc {

// copy Dinv leaves over the diagonal blocks (lower part) : final step of trtri
__global__ void dinv_to_diag_kernel(double* __restrict__ Lbase, long long ld, long long sL,
                                    const double* __restrict__ Dbase, long long sD) {
    const int blk = blockIdx.x, b = blockIdx.z;
    double* L = Lbase + (long long)b * sL + (long long)blk * LEAF * ld + (long long)blk * LEAF;
    const double* D = Dbase + (long long)b * sD + (long long)blk * LEAF * LEAF;
    for (int idx = threadIdx.x; idx < LEAF * LEAF; idx += blockDim.x) {
        const int r = idx >> 7, c = idx & 127;
        if (c <= r) L[(long long)r * ld + c] = D[idx];
    }
}

int current_device() {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= PLMC_MAX_DEVICES) return -1;
    return dev;
}

// function attributes are per device: one flag per device ordinal (idempotent, so a race only repeats the call)
static bool g_leaf_attr_done[PLMC_MAX_DEVICES];
static int leaf_attr() {
    const int dev = current_device();
    if (dev < 0) return PLMC_ERR_LAUNCH;
    if (!g_leaf_attr_done[dev]) {
        if (cudaFuncSetAttribute(potrf_leaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LEAF_SMEM) !=
            cudaSuccess)
            return PLMC_ERR_LAUNCH;
        g_leaf_attr_done[dev] = true;
    }
    return PLMC_OK;
}

// ---------------------------------------------------------------------------
// host-side helpers
// ---------------------------------------------------------------------------
// Split point of the recursions.  Above 512 the matrix is cut at a multiple of 512 so that every diagonal block the
// triangular multiplies treat as a dense leaf starts on a 512 boundary (its zero-padded copy has a fixed slot in
// the side buffer); at and below 512 the cut is at a multiple of the 128-leaf.
static inline int split128(int n) {
    if (n > PB) {   // ... and above 2048 at a multiple of 2048 (the blocks whose inverses the panel solves of potrf use)
        const int k = n / PB;
        return (k >= 2) ? (k / 2) * PB : PB;
    }
    if (n > BLK) {
        const int k = n / BLK;
        return (k >= 2) ? (k / 2) * BLK : BLK;
    }
    return ((n / LEAF) / 2) * LEAF;
}

// lower part of an n x n block (n <= 2048) -> its slot (row stride 2048), zeros above the diagonal
__global__ void tril_copy_kernel(const double* __restrict__ Lbase, long long ld, long long sL,
                                 double* __restrict__ Dbase, long long sD, int n) {
    const int b = blockIdx.z;
    const double* L = Lbase + (long long)b * sL;
    double* D = Dbase + (long long)b * sD;
    const int r = blockIdx.y;
    for (int c = threadIdx.x + blockIdx.x * blockDim.x; c < n; c += blockDim.x * gridDim.x)
        D[(long long)r * PB + c] = (c <= r) ? L[(long long)r * ld + c] : 0.0;
}

// lower part of each diagonal 512-block of L (zero above the diagonal, zero padding up to 512) -> its dense slot
__global__ void dense_diag_copy_kernel(const double* __restrict__ Lbase, long long ld, long long sL,
                                       double* __restrict__ Dbase, long long sD, int n) {
    const int blk = blockIdx.x, b = blockIdx.z;
    const int r0 = blk * BLK;
    const int sz = min(BLK, n - r0);
    const double* L = Lbase + (long long)b * sL + (long long)r0 * ld + r0;
    double* D = Dbase + (long long)b * sD + (long long)blk * BLK * BLK;
    for (int idx = threadIdx.x + blockIdx.y * blockDim.x; idx < BLK * BLK; idx += blockDim.x * gridDim.y) {
        const int r = idx / BLK, c = idx - r * BLK;
        D[idx] = (r < sz && c <= r) ? L[(long long)r * ld + c] : 0.0;
    }
}

static void dense_diag_copy(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0) {
    if (cx.status || n <= 0) return;
    BMat d = D.dense(blk0);
    dim3 grid((n + BLK - 1) / BLK, 8, cx.batch);
    dense_diag_copy_kernel<<<grid, 256, 0, cx.st>>>(L.p, L.ld, L.stride, d.p, d.stride, n);
    if (cudaGetLastError() != cudaSuccess) cx.status = PLMC_ERR_LAUNCH;
    note_launch(1);
}

// ---- optional per-shape timing of every GEMM of the recursion (plmc_trace_enable / plmc_trace_report):
// CUDA events around each launch, aggregated by (path, M, N, K, lower, batch) at report time.
struct TraceRec { int path, M, N, K, lower, batch; cudaEvent_t e0, e1; };
static bool g_trace = false;
static std::vector<TraceRec> g_trace_recs;

static void gemm_impl(LaCtx& cx, bool aKC, bool bKC, BMat A, BMat B, BMat C, int M, int N, int K, double alpha,
                      double beta, int lower, int triA, int triB, int* path);

static void gemm(LaCtx& cx, bool aKC, bool bKC, BMat A, BMat B, BMat C, int M, int N, int K, double alpha,
                 double beta, int lower = 0, int triA = 0, int triB = 0) {
    int path = 0;
    if (!g_trace) { gemm_impl(cx, aKC, bKC, A, B, C, M, N, K, alpha, beta, lower, triA, triB, &path); return; }
    TraceRec r{0, M, N, K, lower, cx.batch, nullptr, nullptr};
    cudaEventCreate(&r.e0); cudaEventCreate(&r.e1);
    cudaEventRecord(r.e0, cx.st);
    gemm_impl(cx, aKC, bKC, A, B, C, M, N, K, alpha, beta, lower, triA, triB, &r.path);
    cudaEventRecord(r.e1, cx.st);
    g_trace_recs.push_back(r);
}

void trace_enable(bool on) { g_trace = on; }

void trace_report() {
    cudaDeviceSynchronize();
    struct Agg { long long count = 0; double ms = 0, flop = 0; };
    std::map<std::array<int, 6>, Agg> agg;
    for (auto& r : g_trace_recs) {
        float ms = 0;
        cudaEventElapsedTime(&ms, r.e0, r.e1);
        Agg& a = agg[{r.path, r.M, r.N, r.K, r.lower, r.batch}];
        a.count++; a.ms += ms;
        a.flop += 2.0 * r.M * r.N * r.K * r.batch * (r.lower ? 0.5 : 1.0) * (r.path == 2 ? 0.5 : 1.0);
        cudaEventDestroy(r.e0); cudaEventDestroy(r.e1);
    }
    g_trace_recs.clear();
    fprintf(stderr, "path      M      N      K lower batch   count   total_ms  TFLOP/s\n");
    for (auto& kv : agg)
        fprintf(stderr, "%-5s %6d %6d %6d %5d %5d %7lld %10.2f %8.1f\n",
                kv.first[0] == 2 ? "tri" : (kv.first[0] ? "int8" : "dmma"), kv.first[1],
                kv.first[2], kv.first[3], kv.first[4], kv.first[5], kv.second.count, kv.second.ms,
                kv.second.flop / kv.second.ms / 1e9);
}

// Which kernel a product takes: 0 FP64 DMMA, 1 INT8 digit planes (*prec slices), 2 INT8 residue planes (*prec moduli).
// The INT8 paths convert their operands to planes BEFORE the product kernel runs, so C may alias A or B for any K;
// the DMMA kernel is in-place safe only when K is a single 128-tile.
static int gemm_route(const LaCtx& cx, int M, int N, int K, bool same, bool tri, int* prec) {
    if (cx.oz_mode <= 0 || cx.oz_prec <= 0 || tri || M < cx.oz_min || N < cx.oz_min || K < cx.oz_min ||
        (long long)M * N * K < cx.oz_min_mnk)
        return 0;
    *prec = cx.oz_prec;
    if (cx.oz_mode == 2) {
        if (!(cx.oz_alt > 0 && (K < cx.oz_rns_min_k || (long long)M * N * K < cx.oz_rns_min_mnk))) return 2;
        *prec = cx.oz_alt;   // short inner dimension / little work: digit planes have the lower per-element cost
    }
    return (ozaki_ws_bytes(M, N, K, *prec, same) + 1024 <= cx.oz_bytes) ? 1 : 0;
}

static void gemm_impl(LaCtx& cx, bool aKC, bool bKC, BMat A, BMat B, BMat C, int M, int N, int K, double alpha,
                      double beta, int lower, int triA, int triB, int* path) {
    if (cx.status) return;
    {
        // large update: FP64 product through the INT8 tensor path (all batch members per launch when
        // the plane scratch holds them, otherwise in passes; everything is ordered on the one stream)
        const bool same = (A.p == B.p && A.ld == B.ld && aKC == bKC && M == N);
        int prec = 0;
        const int route = gemm_route(cx, M, N, K, same, triA || triB, &prec);
        if (route == 2) {   // residue planes: a product that does not fit the scratch is split inside
            cx.status = rns_gemm(aKC, bKC, A.p, A.ld, A.stride, B.p, B.ld, B.stride, C.p, C.ld, C.stride, M, N, K, alpha,
                                 beta, lower, cx.oz_prec, same, cx.batch, cx.oz_ws, cx.oz_bytes, cx.oz_flags, cx.st);
            *path = 1;
            return;
        }
        if (route == 1) {
            cx.status = ozaki_gemm(aKC, bKC, A.p, A.ld, A.stride, B.p, B.ld, B.stride, C.p, C.ld, C.stride, M, N, K,
                                   alpha, beta, lower, prec, same, cx.batch, cx.oz_ws, cx.oz_bytes, cx.st);
            *path = 1;
            return;
        }
    }
    GemmArgs g;
    g.A = A.p; g.B = B.p; g.C = C.p;
    g.lda = A.ld; g.ldb = B.ld; g.ldc = C.ld;
    g.sA = A.stride; g.sB = B.stride; g.sC = C.stride;
    g.M = M; g.N = N; g.K = K;
    g.alpha = alpha; g.beta = beta;
    g.lower = lower; g.triA = triA; g.triB = triB;
    cx.status = gemm_launch(aKC, bKC, g, cx.batch, cx.st);
}

static void trtri_rec(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0);
static bool tri_product(LaCtx& cx, int mode, BMat X, int n, BMat B, BMat C, int m, double alpha);

// blocks of order <= 2048: the plain recursion (solves against 128-leaves)
static void potrf_rec(LaCtx& cx, BMat A, int n, DinvBuf D, long long blk0, int* info) {
    if (cx.status || n <= 0) return;
    if (n == LEAF) {
        if ((cx.status = leaf_attr())) return;
        BMat d = D.leaf(blk0);
        potrf_leaf_kernel<<<cx.batch, LEAF_THREADS, LEAF_SMEM, cx.st>>>(A.p, A.ld, A.stride, d.p, d.stride, info,
                                                                        (int)(blk0 * LEAF));
        if (cudaGetLastError() != cudaSuccess) cx.status = PLMC_ERR_LAUNCH;
        note_launch(1);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat A11 = A, A21 = A.sub(n1, 0), A22 = A.sub(n1, n1);
    potrf_rec(cx, A11, n1, D, blk0, info);
    trsm_rlt(cx, A11, n1, D, blk0, A21, n2, 1.0);
    // A22 -= A21 * A21^T   (lower tiles only)
    gemm(cx, true, true, A21, A21, A22, n2, n2, n1, -1.0, 1.0, /*lower=*/1);
    potrf_rec(cx, A22, n2, D, blk0 + n1 / LEAF, info);
}

// Panel solve of the factorisation, X L^T = alpha B.  In residue mode potrf keeps the explicit inverse of every
// diagonal 2048-block of L it has finished (side buffer, D.panel): the solve against such a block is then ONE
// triangular product X = alpha B inv(L_kk)^T on the tensor path (rns_trmm mode 5) instead of a recursion to sixteen
// 128-leaf products and fifteen updates with K = 128 ... 1024, which ran at 4-56 TFLOP/s-equivalent and made up
// ~400 ms of the C2 iteration.  Between the blocks the update B2 -= X1 L21^T is a plain GEMM as before.
static bool panel_inverses(const LaCtx& cx) { return cx.oz_mode == 2 && cx.oz_prec > 0 && !(cx.oz_flags & 2); }

static void trsm_panel(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (n <= PB) {
        if (n == PB && (blk0 % 16) == 0 && panel_inverses(cx) && tri_product(cx, 5, D.panel(blk0), n, B, B, m, alpha))
            return;
        trsm_rlt(cx, L, n, D, blk0, B, m, alpha);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(0, n1);
    trsm_panel(cx, L, n1, D, blk0, B1, m, alpha);
    gemm(cx, true, true, B1, L.sub(n1, 0), B2, m, n2, n1, -1.0, alpha);
    trsm_panel(cx, L.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m, 1.0);
}

// need_inv: some panel solve further up will use the inverse of the diagonal 2048-blocks of this part
static void potrf_top(LaCtx& cx, BMat A, int n, DinvBuf D, long long blk0, int* info, bool need_inv) {
    if (cx.status || n <= 0) return;
    if (n <= PB) {
        potrf_rec(cx, A, n, D, blk0, info);
        if (need_inv && n == PB && (blk0 % 16) == 0 && panel_inverses(cx) && !cx.status) {
            BMat T = D.panel(blk0);
            tril_copy_kernel<<<dim3(4, n, cx.batch), 256, 0, cx.st>>>(A.p, A.ld, A.stride, T.p, T.stride, n);
            if (cudaGetLastError() != cudaSuccess) { cx.status = PLMC_ERR_LAUNCH; return; }
            note_launch(1);
            trtri_rec(cx, T, n, D, blk0);       // (a failed pivot leaves garbage here as in L: info tells the caller)
        }
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat A11 = A, A21 = A.sub(n1, 0), A22 = A.sub(n1, n1);
    potrf_top(cx, A11, n1, D, blk0, info, true);
    trsm_panel(cx, A11, n1, D, blk0, A21, n2, 1.0);
    // A22 -= A21 * A21^T   (lower tiles only)
    gemm(cx, true, true, A21, A21, A22, n2, n2, n1, -1.0, 1.0, /*lower=*/1);
    potrf_top(cx, A22, n2, D, blk0 + n1 / LEAF, info, need_inv);
}

void potrf_lower(LaCtx& cx, BMat A, int n, DinvBuf D, long long blk0, int* info) {
    potrf_top(cx, A, n, D, blk0, info, false);
}

// X L^T = alpha B ;  L^T = [[L11^T, L21^T],[0, L22^T]]
void trsm_rlt(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (n == LEAF) {  // X = alpha * B * Dinv^T
        gemm(cx, true, true, B, D.leaf(blk0), B, m, LEAF, LEAF, alpha, 0.0);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(0, n1);
    trsm_rlt(cx, L, n1, D, blk0, B1, m, alpha);
    // B2 = alpha*B2 - X1 * L21^T
    gemm(cx, true, true, B1, L.sub(n1, 0), B2, m, n2, n1, -1.0, alpha);
    trsm_rlt(cx, L.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m, 1.0);
}

// X L = alpha B ;  X2 first
void trsm_rln(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (n == LEAF) {  // X = alpha * B * Dinv
        gemm(cx, true, false, B, D.leaf(blk0), B, m, LEAF, LEAF, alpha, 0.0);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(0, n1);
    trsm_rln(cx, L.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m, alpha);
    // B1 = alpha*B1 - X2 * L21
    gemm(cx, true, false, B2, L.sub(n1, 0), B1, m, n1, n2, -1.0, alpha);
    trsm_rln(cx, L, n1, D, blk0, B1, m, 1.0);
}

// L X = alpha B
void trsm_lln(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (n == LEAF) {  // X = alpha * Dinv * B
        gemm(cx, true, false, D.leaf(blk0), B, B, LEAF, m, LEAF, alpha, 0.0);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(n1, 0);
    trsm_lln(cx, L, n1, D, blk0, B1, m, alpha);
    // B2 = alpha*B2 - L21 * X1
    gemm(cx, true, false, L.sub(n1, 0), B1, B2, n2, m, n1, -1.0, alpha);
    trsm_lln(cx, L.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m, 1.0);
}

// L^T X = alpha B ;  X2 first
void trsm_llt(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (n == LEAF) {  // X = alpha * Dinv^T * B
        gemm(cx, false, false, D.leaf(blk0), B, B, LEAF, m, LEAF, alpha, 0.0);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(n1, 0);
    trsm_llt(cx, L.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m, alpha);
    // B1 = alpha*B1 - L21^T * X2
    gemm(cx, false, false, L.sub(n1, 0), B2, B1, n1, m, n2, -1.0, alpha);
    trsm_llt(cx, L, n1, D, blk0, B1, m, 1.0);
}

// ---- triangular multiplies with DENSE 512-leaves -----------------------------------------------------------
// A triangular solve needs the inverse of its diagonal blocks, so its recursion has to go down to the 128-leaf
// whose inverse the Cholesky leaf emitted: n/128 tall-skinny K = 128 products per solve, FP64-pipe bound at
// 15-20 TFLOP/s (the "tail" of round 1).  A triangular MULTIPLY has no such constraint: its diagonal block can
// simply be treated as dense (zero above the diagonal) at any size.  The inverse is therefore organised as
//     inv(L) = [[X11, 0], [-X22 L21 X11, X22]]   with X11, X22 inverted FIRST,
// i.e. two triangular multiplies per level instead of two solves, and both they and the L^T L product stop their
// recursion at 512: the leaf is one K = 512 GEMM on the tensor path against the zero-padded dense copy of the
// diagonal block kept in the side buffer (2-7 % more flops, none of them on the FP64 pipe).
// A dense leaf is taken only when the product goes to an INT8 kernel (operands are converted to planes before the
// product runs, so updating B in place is safe); otherwise the recursion continues to the 128-leaf on DMMA.
static bool dense_leaf(const LaCtx& cx, int M, int N, int K) {
    int prec = 0;
    return gemm_route(cx, M, N, K, false, false, &prec) != 0;
}

// A product with a lower-triangular operand of order n as ONE residue-plane launch set whose INT8 GEMM visits
// only the k-tiles that can be nonzero (rns_trmm, csrc/ozaki2.cu) -- instead of the recursion below, which cuts it into
// n/512 leaf products with K = 512 and updates of every size above that (43-80 TFLOP/s-equivalent at C2 against
// 150+ for a product that runs its whole inner dimension in one pass).  mode: 1 B X, 2 X B, 3 X^T B, 4 X^T X (lower).
// Taken in residue mode when the order reaches the residue scheme's minimum inner dimension and the (triangular) work
// its minimum; returns false when the product should take the recursion (also when the scratch cannot hold it).
// mode 5: B X^T (the panel solve of potrf with X = the inverse of a diagonal block).
static bool tri_product(LaCtx& cx, int mode, BMat X, int n, BMat B, BMat C, int m, double alpha) {
    if (cx.oz_mode != 2 || cx.oz_prec <= 0 || (cx.oz_flags & 4)) return false;
    const int kmin = cx.oz_rns_min_k > BLK ? cx.oz_rns_min_k : BLK;
    const double work = (mode == 4) ? (double)n * n * n / 3.0 : (double)m * n * n / 2.0;
    // mode 5 (panel solve of potrf): the alternative is a solve recursion, not a digit-plane GEMM -- a quarter of the
    // residue scheme's work floor is enough
    const double floor_rns = (mode == 5) ? (double)cx.oz_rns_min_mnk * 0.25 : (double)cx.oz_rns_min_mnk;
    if (n < kmin || (mode != 4 && m < cx.oz_min) || work < floor_rns || work < (double)cx.oz_min_mnk) return false;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (g_trace) {
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaEventRecord(e0, cx.st);
    }
    const int rc = rns_trmm(mode, X.p, X.ld, X.stride, B.p, B.ld, B.stride, C.p, C.ld, C.stride, n, m, alpha, 0.0,
                            cx.oz_prec, cx.batch, cx.oz_ws, cx.oz_bytes, cx.oz_flags, cx.st);
    if (g_trace) {
        if (rc == 0) {
            cudaEventRecord(e1, cx.st);
            const int M = (mode == 1 || mode == 5) ? m : n, N = (mode == 1 || mode == 4 || mode == 5) ? n : m;
            g_trace_recs.push_back(TraceRec{2, M, N, n, mode == 4 ? 1 : 0, cx.batch, e0, e1});
        } else {
            cudaEventDestroy(e0); cudaEventDestroy(e1);
        }
    }
    if (rc == 1) return false;      // does not fit the scratch: recurse (the halves will)
    if (rc != 0) cx.status = rc;
    return true;
}

// B := alpha * B * X   (X lower n x n, B m x n)
static void trmm_rln(LaCtx& cx, BMat X, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (tri_product(cx, 1, X, n, B, B, m, alpha)) return;
    if (n <= BLK && (blk0 % 4) == 0 && dense_leaf(cx, m, n, n)) {
        gemm(cx, true, false, B, D.dense(blk0), B, m, n, n, alpha, 0.0);
        return;
    }
    if (n == LEAF) {
        gemm(cx, true, false, B, X, B, m, LEAF, LEAF, alpha, 0.0, 0, 0, /*triB=*/1);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(0, n1);
    trmm_rln(cx, X, n1, D, blk0, B1, m, alpha);                                   // B1 := a B1 Xa
    gemm(cx, true, false, B2, X.sub(n1, 0), B1, m, n1, n2, alpha, 1.0);           // B1 += a B2 Xc
    trmm_rln(cx, X.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m, alpha);           // B2 := a B2 Xb
}

// B := alpha * X * B   (X lower n x n, B n x m)
static void trmm_lln(LaCtx& cx, BMat X, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (tri_product(cx, 2, X, n, B, B, m, alpha)) return;
    if (n <= BLK && (blk0 % 4) == 0 && dense_leaf(cx, n, m, n)) {
        gemm(cx, true, false, D.dense(blk0), B, B, n, m, n, alpha, 0.0);
        return;
    }
    if (n == LEAF) {
        gemm(cx, true, false, X, B, B, LEAF, m, LEAF, alpha, 0.0, 0, /*triA=*/1, 0);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(n1, 0);
    trmm_lln(cx, X.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m, alpha);           // B2 := a Xb B2
    gemm(cx, true, false, X.sub(n1, 0), B1, B2, n2, m, n1, alpha, 1.0);           // B2 += a Xc B1
    trmm_lln(cx, X, n1, D, blk0, B1, m, alpha);                                   // B1 := a Xa B1
}

// blocks of order <= 512: L21 := -inv(L22) L21 inv(L11) by two solves on the not-yet-inverted diagonal blocks
static void trtri_small(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0) {
    if (cx.status || n <= LEAF) return;
    const int n1 = split128(n), n2 = n - n1;
    BMat L21 = L.sub(n1, 0), L22 = L.sub(n1, n1);
    trsm_rln(cx, L, n1, D, blk0, L21, n2, 1.0);
    trsm_lln(cx, L22, n2, D, blk0 + n1 / LEAF, L21, n1, -1.0);
    trtri_small(cx, L, n1, D, blk0);
    trtri_small(cx, L22, n2, D, blk0 + n1 / LEAF);
}

static void trtri_rec(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0) {
    if (cx.status || n <= 0) return;
    if (n <= BLK) {
        trtri_small(cx, L, n, D, blk0);
        if (cx.status) return;
        dim3 grid(n / LEAF, 1, cx.batch);
        BMat d0 = D.leaf(blk0);
        dinv_to_diag_kernel<<<grid, 256, 0, cx.st>>>(L.p, L.ld, L.stride, d0.p, d0.stride);
        if (cudaGetLastError() != cudaSuccess) cx.status = PLMC_ERR_LAUNCH;
        note_launch(1);
        if ((blk0 % 4) == 0) dense_diag_copy(cx, L, n, D, blk0);   // the inverted block, for the multiplies above
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat L21 = L.sub(n1, 0), L22 = L.sub(n1, n1);
    trtri_rec(cx, L, n1, D, blk0);
    trtri_rec(cx, L22, n2, D, blk0 + n1 / LEAF);
    // L21 := -X22 (L21 X11)
    trmm_rln(cx, L, n1, D, blk0, L21, n2, 1.0);
    trmm_lln(cx, L22, n2, D, blk0 + n1 / LEAF, L21, n1, -1.0);
}

// B := alpha X B for a lower-triangular X; the dense copies of X's diagonal 512-blocks are (re)written first
void trmm_lln_lower(LaCtx& cx, BMat X, int n, DinvBuf D, BMat B, int m, double alpha, bool fill_dense) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (fill_dense) dense_diag_copy(cx, X, n, D, 0);
    trmm_lln(cx, X, n, D, 0, B, m, alpha);
}

// op 1: B := alpha B X (B m x n) | 2: B := alpha X B | 3: B := X^T B (alpha must be 1)   (B n x m for 2, 3)
void trmm_lower(LaCtx& cx, int op, BMat X, int n, DinvBuf D, BMat B, int m, double alpha) {
    if (cx.status || n <= 0 || m <= 0) return;
    dense_diag_copy(cx, X, n, D, 0);
    if (op == 1) trmm_rln(cx, X, n, D, 0, B, m, alpha);
    else if (op == 2) trmm_lln(cx, X, n, D, 0, B, m, alpha);
    else trmm_llt(cx, X, n, D, 0, B, m);
}

void trtri_lower(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0) {
    if (cx.status || n <= 0) return;
    trtri_rec(cx, L, n, D, blk0);
}

// B := T^T B
void trmm_llt(LaCtx& cx, BMat T, int n, DinvBuf D, long long blk0, BMat B, int m) {
    if (cx.status || n <= 0 || m <= 0) return;
    if (tri_product(cx, 3, T, n, B, B, m, 1.0)) return;
    if (n <= BLK && (blk0 % 4) == 0 && dense_leaf(cx, n, m, n)) {
        gemm(cx, false, false, D.dense(blk0), B, B, n, m, n, 1.0, 0.0);
        return;
    }
    if (n == LEAF) {
        gemm(cx, false, false, T, B, B, LEAF, m, LEAF, 1.0, 0.0, 0, /*triA=*/1, 0);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat B1 = B, B2 = B.sub(n1, 0);
    trmm_llt(cx, T, n1, D, blk0, B1, m);
    // B1 += T21^T * B2
    gemm(cx, false, false, T.sub(n1, 0), B2, B1, n1, m, n2, 1.0, 1.0);
    trmm_llt(cx, T.sub(n1, n1), n2, D, blk0 + n1 / LEAF, B2, m);
}

static void lauum_rec(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0) {
    if (cx.status || n <= 0) return;
    if (tri_product(cx, 4, L, n, L, L, n, 1.0)) return;
    if (n <= BLK && n > LEAF && (blk0 % 4) == 0) {
        // C = T^T T (lower tiles) from the dense copy of the block: operands and result do not alias
        BMat T = D.dense(blk0);
        gemm(cx, false, false, T, T, L, n, n, n, 1.0, 0.0, /*lower=*/1);
        return;
    }
    if (n == LEAF) {  // C = T^T T (full symmetric tile written)
        gemm(cx, false, false, L, L, L, LEAF, LEAF, LEAF, 1.0, 0.0, 0, 1, 1);
        return;
    }
    const int n1 = split128(n), n2 = n - n1;
    BMat L21 = L.sub(n1, 0), L22 = L.sub(n1, n1);
    lauum_rec(cx, L, n1, D, blk0);
    // L11 += L21^T L21  (lower tiles)
    gemm(cx, false, false, L21, L21, L, n1, n1, n2, 1.0, 1.0, /*lower=*/1);
    // L21 := L22^T L21
    trmm_llt(cx, L22, n2, D, blk0 + n1 / LEAF, L21, n1);
    lauum_rec(cx, L22, n2, D, blk0 + n1 / LEAF);
}

void lauum_lower(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, bool fill_dense) {
    if (cx.status || n <= 0) return;
    if (fill_dense) dense_diag_copy(cx, L, n, D, blk0);
    lauum_rec(cx, L, n, D, blk0);
}

// lower(C) := alpha A^T A + beta C  (A k x n): one routed product, the operand is converted once (same_operand)
void syrk_lower(LaCtx& cx, BMat A, int n, int k, BMat C, double alpha, double beta) {
    if (cx.status || n <= 0 || k <= 0) return;
    gemm(cx, false, false, A, A, C, n, n, k, alpha, beta, /*lower=*/1);
}

}  // namespace plmc
