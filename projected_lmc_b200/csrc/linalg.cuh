// Batched blocked dense linear algebra on top of the DMMA GEMM.
//
// Every routine is a recursive (cache-oblivious) block algorithm whose leaves
// are 128x128: all O(n^3) work is done by gemm_dmma_kernel; the only other
// compute kernel on the factorisation path is the 128x128 shared-memory
// Cholesky leaf, which also emits the explicit inverse of its factor (Dinv) so
// that every triangular-solve leaf is again a GEMM.
//
// All matrices: row-major, order n % 128 == 0, batch via stride.
#pragma once
#include "gemm_dmma.cuh"

namespace plmc {

struct BMat {  // batched matrix view
    double* p;
    long long ld;
    long long stride;
    __host__ BMat sub(long long r, long long c) const { return BMat{p + r * ld + c, ld, stride}; }
};

struct LaCtx {
    cudaStream_t st;
    int batch;
    int status;  // first non-zero launch status
    // FP64 through the INT8 tensor path (tcgen05) for the large GEMMs of the recursion (plmc_gemm_cfg):
    // mode 0 = off (DMMA only), 1 = digit planes (csrc/ozaki.cu, oz_prec slices), 2 = residue planes
    // (csrc/ozaki2.cu, oz_prec moduli)
    void* oz_ws = nullptr;
    long long oz_bytes = 0;
    int oz_mode = 0;
    int oz_prec = 0;
    int oz_min = 1024;  // smallest M, N, K routed to the INT8 path
    long long oz_min_mnk = 0;   // and the least work M*N*K
    int oz_flags = 0;   // bit 0: single-CTA kernel in mode 2
    // mode 2: digit planes (oz_alt slices) for products with K < oz_rns_min_k or M N K < oz_rns_min_mnk
    int oz_alt = 0;
    int oz_rns_min_k = 0;
    long long oz_rns_min_mnk = 0;
};

// per-device one-time state (function attributes, SM count): indexed by the CUDA device ordinal
constexpr int PLMC_MAX_DEVICES = 64;
int current_device();   // -1 on failure

int trsv_solve(const double* L, long long ld, long long sL, const double* dinv, long long sD, const double* y,
               long long ldy, double* v, long long sV, double* z, double* alpha, long long ldv, long long n,
               long long npad, int batch, cudaStream_t st);

void trace_enable(bool on);
void trace_report();

long long ozaki_ws_bytes(int M, int N, int K, int s, bool same_operand);
int ozaki_gemm(bool aKC, bool bKC, const double* A, long long lda, long long sA, const double* B, long long ldb,
               long long sB, double* C, long long ldc, long long sC, int M, int N, int K, double alpha, double beta,
               int lower, int s, bool same_operand, int batch, void* ws, long long ws_bytes, cudaStream_t st);

int rns_bits(int nmod, int K);
long long rns_ws_bytes(int M, int N, int K, int nmod, bool same_operand, bool lower);
int rns_gemm(bool aKC, bool bKC, const double* A, long long lda, long long sA, const double* B, long long ldb,
             long long sB, double* C, long long ldc, long long sC, int M, int N, int K, double alpha, double beta,
             int lower, int nmod, bool same_operand, int batch, void* ws, long long ws_bytes, int flags,
             cudaStream_t st);

// products with a lower-triangular operand X (order n) in one launch set (csrc/ozaki2.cu); returns 1 if the scratch
// does not hold one batch member (nothing launched), else a PLMC_* status
int rns_trmm(int mode, const double* X, long long ldx, long long sX, const double* B, long long ldb, long long sB,
             double* C, long long ldc, long long sC, int n, int m, double alpha, double beta, int nmod, int batch,
             void* ws, long long ws_bytes, int flags, cudaStream_t st);

// Side buffer of the factorisation layer, per batch member (stride = dinv_elems(npad)):
//   [0, npad*128)            n/128 consecutive 128x128 row-major blocks holding inv(L_kk) of the 128-leaves
//                            (upper part explicitly zero), written by potrf;
//   [npad*128, ...)          ceil(npad/512) slots of 512x512: zero-padded DENSE copies of the diagonal 512-blocks of
//                            the triangular matrix being multiplied (trtri / lauum), so that the leaf of a
//                            triangular multiply is one K = 512 GEMM on the tensor path instead of a 128-recursion.
//   [.., ...)                ceil(npad/2048) slots of 2048x2048: explicit inverses of the diagonal 2048-blocks of L,
//                            written by potrf as it goes (residue mode): the panel solve against such a block is ONE
//                            triangular product on the tensor path instead of a solve recursion to the 128-leaves.
constexpr int BLK = 512;
constexpr int PB = 2048;
__host__ inline long long dinv_elems(long long npad) {   // (no 2048-slots for matrices that are a single panel block)
    return npad * 128 + ((npad + BLK - 1) / BLK) * (long long)BLK * BLK +
           (npad > PB ? ((npad + PB - 1) / PB) * (long long)PB * PB : 0);
}
struct DinvBuf {
    double* p;
    long long stride;
    long long dense_off;   // npad * 128
    long long panel_off;   // dense_off + ceil(npad/512) * 512^2
    __host__ BMat leaf(long long blk) const { return BMat{p + blk * 16384, 128, stride}; }
    // dense copy of the 512-block that starts at 128-leaf index blk (blk % 4 == 0)
    __host__ BMat dense(long long blk) const { return BMat{p + dense_off + (blk / 4) * (long long)BLK * BLK, BLK, stride}; }
    // inverse of the diagonal 2048-block that starts at 128-leaf index blk (blk % 16 == 0)
    __host__ BMat panel(long long blk) const { return BMat{p + panel_off + (blk / 16) * (long long)PB * PB, PB, stride}; }
};
__host__ inline DinvBuf make_dinv(const double* dinv, long long npad) {
    const long long dense_off = npad * 128;
    return DinvBuf{const_cast<double*>(dinv), dinv_elems(npad), dense_off,
                   dense_off + ((npad + BLK - 1) / BLK) * (long long)BLK * BLK};
}

// A (lower) -> L in place; info[b] = 0 or 1-based index of first non-positive pivot.
void potrf_lower(LaCtx& cx, BMat A, int n, DinvBuf D, long long blk0, int* info);
// X * L^T = alpha*B    (B: m x n, in place)
void trsm_rlt(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha);
// X * L = alpha*B
void trsm_rln(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha);
// L * X = alpha*B      (B: n x m, in place)
void trsm_lln(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha);
// L^T * X = alpha*B
void trsm_llt(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, BMat B, int m, double alpha);
// L -> inv(L) in place (needs Dinv from potrf_lower); leaves dense copies of the inverted 512-blocks in D
void trtri_lower(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0);
// L -> lower(L^T L) in place; D supplies (and, with fill_dense, receives) the dense copies of L's diagonal blocks
void lauum_lower(LaCtx& cx, BMat L, int n, DinvBuf D, long long blk0, bool fill_dense);
// B := alpha * X * B  (X lower n x n, B n x m): triangular multiply with dense 512-leaves; fill_dense refreshes
// the dense copies of X's diagonal blocks in D first (not needed right after trtri_lower on the same matrix)
void trmm_lln_lower(LaCtx& cx, BMat X, int n, DinvBuf D, BMat B, int m, double alpha, bool fill_dense);
// op 1: B := alpha B X (B m x n) | 2: B := alpha X B | 3: B := X^T B (alpha = 1)  (B n x m); refreshes the dense copies
void trmm_lower(LaCtx& cx, int op, BMat X, int n, DinvBuf D, BMat B, int m, double alpha);
// B := T^T * B  (T lower n x n, B n x m)
void trmm_llt(LaCtx& cx, BMat T, int n, DinvBuf D, long long blk0, BMat B, int m);
// lower(C) := alpha * A^T A + beta * C  (A k x n, C n x n), routed like every product of the recursions
void syrk_lower(LaCtx& cx, BMat A, int n, int k, BMat C, double alpha, double beta);

}  // namespace plmc
