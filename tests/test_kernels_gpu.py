"""GPU: every C-ABI entry point against torch float64 on the same device / the CPU oracle,
including ragged shapes, failure reporting and size-independent properties at large n."""
import math

import pytest
import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import ops

from .helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rnd(*shape, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(*shape, generator=g, dtype=torch.float64).to(DEV)


def spd(b, n, seed=0):
    X = rnd(b, n, n + 32, seed=seed)
    return X @ X.transpose(1, 2) / n + torch.eye(n, dtype=torch.float64, device=DEV)


@pytest.mark.parametrize("layout", [0, 1, 2, 3])
@pytest.mark.parametrize("alpha,beta", [(1.0, 0.0), (-0.5, 1.0), (2.0, -0.25)])
def test_gemm_layouts(layout, alpha, beta):
    M, N, K, b = 256, 384, 160, 3
    a_mc, b_nc = bool(layout & 2), bool(layout & 1)
    A = rnd(b, K, M, seed=1) if a_mc else rnd(b, M, K, seed=1)
    B = rnd(b, K, N, seed=2) if b_nc else rnd(b, N, K, seed=2)
    C = rnd(b, M, N, seed=3)
    opA = A.transpose(1, 2) if a_mc else A
    opB = B if b_nc else B.transpose(1, 2)
    ref = alpha * opA @ opB + beta * C
    ops.gemm(layout, A, B, C, M, N, K, alpha=alpha, beta=beta)
    assert (C - ref).abs().max().item() < 1e-11


def test_gemm_beta_zero_ignores_nan_in_c():
    A, B = rnd(1, 128, 128, seed=1), rnd(1, 128, 128, seed=2)
    C = torch.full((1, 128, 128), float("nan"), dtype=torch.float64, device=DEV)
    ops.gemm(0, A, B, C, 128, 128, 128)
    assert torch.isfinite(C).all()


def test_gemm_lower_only_and_triangular_masks():
    n = 384
    P = rnd(2, n, 256, seed=4)
    C0 = rnd(2, n, n, seed=5)
    C = C0.clone()
    ops.gemm(0, P, P, C, n, n, 256, alpha=-1.0, beta=1.0, lower=True)
    ref = C0 - P @ P.transpose(1, 2)
    for i in range(3):
        for j in range(3):
            blk = (slice(None), slice(128 * i, 128 * i + 128), slice(128 * j, 128 * j + 128))
            if i >= j:
                assert (C[blk] - ref[blk]).abs().max().item() < 1e-11
            else:
                assert torch.equal(C[blk], C0[blk])           # strictly-upper tiles untouched
    # triangular operands: garbage (NaN) above the diagonal must never be read
    T = rnd(1, 128, 128, seed=6)
    Tn = T.clone()
    Tn[0][torch.triu(torch.ones(128, 128, dtype=torch.bool, device=DEV), 1)] = float("nan")
    Bm = rnd(1, 128, 256, seed=7)
    out = torch.empty_like(Bm)
    ops.gemm(3, Tn, Bm, out, 128, 256, 128, triA=True)        # out = tril(T)^T @ B
    assert (out - torch.tril(T).transpose(1, 2) @ Bm).abs().max().item() < 1e-11
    out2 = torch.empty(1, 128, 128, dtype=torch.float64, device=DEV)
    ops.gemm(3, Tn, Tn, out2, 128, 128, 128, triA=True, triB=True)   # tril(T)^T tril(T)
    assert (out2 - torch.tril(T).transpose(1, 2) @ torch.tril(T)).abs().max().item() < 1e-11


@pytest.mark.parametrize("n,b", [(128, 1), (256, 5), (640, 2), (1152, 3)])
def test_potrf_solve_trtri_lauum(n, b):
    K0 = spd(b, n, seed=n)
    K = K0.clone()
    dinv = ops.alloc_dinv(n, b, DEV)
    info = torch.full((b,), 7, dtype=torch.int32, device=DEV)
    ops.potrf(K, dinv, info)
    assert info.tolist() == [0] * b
    Lref = torch.linalg.cholesky(K0)
    assert (torch.tril(K) - Lref).abs().max().item() < 1e-12
    y = rnd(b, n, seed=11)
    z, alpha, quad, logdet = ops.solve_logdet(K, dinv, y, n)
    zref = torch.linalg.solve_triangular(Lref, y.unsqueeze(-1), upper=False).squeeze(-1)
    assert (z - zref).abs().max().item() < 1e-11
    assert (alpha - torch.cholesky_solve(y.unsqueeze(-1), Lref).squeeze(-1)).abs().max().item() < 1e-11
    assert torch.allclose(quad, zref.pow(2).sum(-1), rtol=1e-13)
    assert torch.allclose(logdet, 2 * torch.log(torch.diagonal(Lref, dim1=1, dim2=2)).sum(-1), rtol=1e-13, atol=1e-12)
    ops.trtri(K, dinv)
    assert (torch.tril(K) - torch.linalg.inv(Lref)).abs().max().item() < 1e-11
    ops.lauum(K, dinv)
    assert (torch.tril(K) - torch.tril(torch.linalg.inv(K0))).abs().max().item() < 1e-10


@pytest.mark.parametrize("mode,prec", [(ops.GEMM_INT8_DIGITS, 7), (ops.GEMM_INT8_RNS, 16)])
@pytest.mark.parametrize("n", [1664, 2560])          # 3 x 512 + 128 (ragged last block) and 5 x 512
def test_inverse_with_dense_512_leaves_on_the_tensor_path(mode, prec, n):
    """trtri / lauum as triangular MULTIPLIES whose leaves are K = 512 products against zero-padded dense copies of
    the diagonal blocks (INT8 path, in place), with every product routed to the tensor path (no work floor)."""
    b = 2
    K0 = spd(b, n, seed=n + prec)
    K = K0.clone()
    dinv = ops.alloc_dinv(n, b, DEV)
    info = torch.zeros(b, dtype=torch.int32, device=DEV)
    ws = torch.empty(1 << 30, dtype=torch.uint8, device=DEV)
    cfg = ops.gemm_cfg(ws, mode, prec, min_dim=128, alt_precision=0, min_mnk=0)
    ops.potrf(K, dinv, info, cfg)
    assert info.tolist() == [0] * b
    Lref = torch.linalg.cholesky(K0)
    assert rel_err(torch.tril(K), Lref) < 1e-12
    ops.trtri(K, dinv, cfg)
    assert rel_err(torch.tril(K), torch.linalg.inv(Lref)) < 1e-10
    ops.lauum(K, dinv, cfg)
    assert rel_err(torch.tril(K), torch.tril(torch.linalg.inv(K0))) < 1e-9
    # potri = trtri + lauum in one call gives the same bits
    K2 = K0.clone()
    ops.potrf(K2, dinv, info, cfg)
    ops.potri(K2, dinv, cfg)
    assert torch.equal(torch.tril(K2), torch.tril(K))


@pytest.mark.parametrize("n", [6144, 4736])          # 3 x 2048, and 2 x 2048 + 640 (ragged last block)
def test_potrf_panel_solves_through_the_inverses_of_the_diagonal_2048_blocks(n):
    """Residue mode, default routing thresholds: the panel solve below a finished diagonal 2048-block is one
    triangular product with the block's explicit inverse (rns_trmm mode 5).  Same factor as torch's Cholesky, same
    solves / inverse afterwards, and the diagnostic flag that restores the 128-leaf solves agrees to rounding."""
    b = 2
    K0 = spd(b, n, seed=n)
    Lref = torch.linalg.cholesky(K0)
    ws = torch.empty(6 << 30, dtype=torch.uint8, device=DEV)
    out = {}
    for flags in (0, 2):
        cfg = ops.gemm_cfg(ws, ops.GEMM_INT8_RNS, 15, min_dim=128, flags=flags, alt_precision=7, rns_min_k=1024,
                           rns_min_mnk=int(2e10), min_mnk=512 ** 3)
        K = K0.clone()
        dinv = ops.alloc_dinv(n, b, DEV)
        info = torch.zeros(b, dtype=torch.int32, device=DEV)
        ops.potrf(K, dinv, info, cfg)
        assert info.tolist() == [0] * b
        out[flags] = torch.tril(K).clone()
        assert rel_err(out[flags], Lref) < 1e-12, flags
        y = rnd(b, n, seed=3)
        z, alpha, quad, logdet = ops.solve_logdet(K, dinv, y, n)
        zref = torch.linalg.solve_triangular(Lref, y.unsqueeze(-1), upper=False)
        aref = torch.linalg.solve_triangular(Lref.transpose(1, 2), zref, upper=True).squeeze(-1)
        assert rel_err(alpha, aref) < 1e-10
        ops.potri(K, dinv, cfg)
        assert rel_err(torch.tril(K), torch.tril(torch.linalg.inv(K0))) < 1e-9
    assert rel_err(out[0], out[2]) < 1e-13


def test_potrf_reports_first_bad_pivot_per_batch_member():
    n = 384
    K = spd(3, n, seed=2)
    K[1, 200, 200] = -5.0          # member 1 loses positive definiteness at pivot 201 (1-based)
    K[2, 0, 0] = 0.0               # member 2 fails at the very first pivot
    K0 = K.clone()
    dinv = ops.alloc_dinv(n, 3, DEV)
    info = torch.zeros(3, dtype=torch.int32, device=DEV)
    ops.potrf(K, dinv, info)
    got = info.tolist()
    _, ref_info = torch.linalg.cholesky_ex(K0)
    assert got[0] == 0 and got[1] == ref_info[1].item() == 201 and got[2] == ref_info[2].item() == 1
    assert (torch.tril(K[0]) - torch.linalg.cholesky(K0[0])).abs().max().item() < 1e-12   # healthy member unaffected


@pytest.mark.parametrize("op", [0, 1, 2, 3])
def test_trsm_ops(op):
    n, m, b = 512, 256, 2
    K0 = spd(b, n, seed=3)
    K = K0.clone()
    dinv = ops.alloc_dinv(n, b, DEV)
    info = torch.zeros(b, dtype=torch.int32, device=DEV)
    ops.potrf(K, dinv, info)
    L = torch.tril(K)
    B0 = rnd(b, m, n, seed=5) if op in (0, 1) else rnd(b, n, m, seed=5)
    B = B0.clone()
    ops.trsm(op, K, dinv, B, alpha=-0.5)
    if op == 0:
        ref = torch.linalg.solve_triangular(L.transpose(1, 2), -0.5 * B0, upper=True, left=False)
    elif op == 1:
        ref = torch.linalg.solve_triangular(L, -0.5 * B0, upper=False, left=False)
    elif op == 2:
        ref = torch.linalg.solve_triangular(L, -0.5 * B0, upper=False)
    else:
        ref = torch.linalg.solve_triangular(L.transpose(1, 2), -0.5 * B0, upper=True)
    assert (B - ref).abs().max().item() < 1e-10


@pytest.mark.parametrize("mode,prec", [(None, 0), (ops.GEMM_INT8_DIGITS, 7), (ops.GEMM_INT8_RNS, 16)])
@pytest.mark.parametrize("n,m", [(640, 256), (1664, 1024)])      # ragged last 512-block in both
def test_trmm_with_the_explicit_inverse_equals_the_triangular_solve(mode, prec, n, m):
    """plmc_trmm_batched op 2 (B := a X B, X = inv(L) from trtri): the predictive-variance product as a triangular
    multiply; same result as the solve with L, in pure FP64 (128-leaves) and on the tensor path (dense 512-leaves)."""
    b = 2
    K0 = spd(b, n, seed=n)
    K = K0.clone()
    dinv = ops.alloc_dinv(n, b, DEV)
    info = torch.zeros(b, dtype=torch.int32, device=DEV)
    cfg = None
    if mode is not None:
        ws = torch.empty(1 << 30, dtype=torch.uint8, device=DEV)
        cfg = ops.gemm_cfg(ws, mode, prec, min_dim=128, alt_precision=0, min_mnk=0)
    ops.potrf(K, dinv, info, cfg)
    Lref = torch.linalg.cholesky(K0)
    B0 = rnd(b, n, m, seed=9)
    ref = torch.linalg.solve_triangular(Lref, -0.5 * B0, upper=False)
    Bs = B0.clone()
    ops.trsm(2, K, dinv, Bs, alpha=-0.5, cfg=cfg)
    ops.trtri(K, dinv, cfg)
    K.add_(torch.triu(torch.full_like(K, float("nan")), 1))              # the strict upper part is never read
    Bm = B0.clone()
    ops.trmm(2, K, dinv, Bm, alpha=-0.5, cfg=cfg)
    assert rel_err(Bs, ref) < 1e-11 and rel_err(Bm, ref) < 1e-11
    with pytest.raises(Exception):
        ops.trmm(0, K, dinv, Bm)
    # the other two triangular multiplies (B X and X^T B) against dense products with tril(X)
    Xl = torch.tril(torch.nan_to_num(K, nan=0.0))
    B1 = rnd(b, m, n, seed=10)
    ref1 = 0.75 * B1 @ Xl
    ops.trmm(1, K, dinv, B1, alpha=0.75, cfg=cfg)
    B3 = B0.clone()
    ops.trmm(3, K, dinv, B3, cfg=cfg)
    assert rel_err(B1, ref1) < 1e-12 and rel_err(B3, Xl.transpose(1, 2) @ B0) < 1e-12


@pytest.mark.parametrize("n,p,q", [(1, 1, 1), (63, 7, 4), (1000, 50, 10), (4097, 65, 33), (513, 500, 32), (31, 2, 1),
                                   (777, 6, 3), (5000, 34, 17), (100003, 32, 8), (44484, 8, 4), (20000, 100, 16)])
def test_projection_fwd_bwd(n, p, q):
    Y, T = rnd(n, p, seed=1), rnd(p, q, seed=2)
    TY = ops.project_fwd(Y, T)
    assert TY.shape == (q, n)
    assert (TY - (Y @ T).T).abs().max().item() < 1e-11 * max(1, p)
    G = rnd(q, n, seed=3)
    dT = ops.project_bwd(Y, G)
    assert (dT - Y.T @ G.T).abs().max().item() < 1e-10 * max(1.0, math.sqrt(n))


def _oracle_params(kind, ell, noise, os_=None):
    q, d = ell.shape
    inv = lambda v: v + torch.log(-torch.expm1(-v))          # inverse softplus
    return O.OracleParams(raw_lengthscale=inv(ell.cpu())[:, None, :], raw_noise=inv(noise.cpu())[:, None],
                          noise_lower=0.0, kernel=kind, raw_outputscale=None if os_ is None else inv(os_.cpu()))


@pytest.mark.parametrize("kind,kid", [("rbf", 0), ("matern52", 1), ("matern32", 2), ("matern12", 3)])
@pytest.mark.parametrize("n,d,with_os", [(100, 1, False), (300, 6, True), (257, 21, False)])
def test_gram_and_cross_gram_vs_oracle(kind, kid, n, d, with_os):
    q = 3
    g = torch.Generator().manual_seed(n + d)
    X = (torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1)
    ell = torch.rand(q, d, generator=g, dtype=torch.float64) + 0.4
    noise = torch.rand(q, generator=g, dtype=torch.float64) * 0.3 + 0.05
    os_ = (torch.rand(q, generator=g, dtype=torch.float64) + 0.5) if with_os else None
    Xg, ellg, ng = X.to(DEV), ell.to(DEV), noise.to(DEV)
    osg = None if os_ is None else os_.to(DEV)
    np_ = ops.npad(n)
    Z, zn = ops.scale_inputs(Xg, ops.col_mean(Xg), ellg, np_)
    K = torch.full((q, np_, np_), float("nan"), dtype=torch.float64, device=DEV)
    ops.gram(Z, zn, kid, osg, ng, K, n)
    p = _oracle_params(kind, ell, noise, os_)
    Kref = O.gram(p, X, training=False) + torch.diag_embed(noise[:, None].expand(-1, n))
    low = torch.tril(torch.ones(n, n, dtype=torch.bool))
    got = K[:, :n, :n].cpu()
    tol = 1e-7 if kind == "matern12" else 1e-12       # nu=1/2: sqrt amplifies the expansion's round-off near r=0
    assert (got - Kref)[:, low].abs().max().item() < tol
    # identity padding, lower part
    if np_ > n:
        pad = K[:, n:, :].cpu()
        eye = torch.zeros_like(pad)
        eye[:, torch.arange(np_ - n), n + torch.arange(np_ - n)] = 1.0
        lowpad = torch.tril(torch.ones(np_, np_, dtype=torch.bool))[n:, :]
        assert torch.equal(pad[:, lowpad], eye[:, lowpad])
    # cross Gram against test points
    ns = 150
    Xs = torch.rand(ns, d, generator=g, dtype=torch.float64) * 2 - 1
    mt = ops.npad(ns)
    Zt, znt = ops.scale_inputs(Xs.to(DEV), ops.col_mean(Xg), ellg, mt)
    Kx = torch.empty((q, np_, mt), dtype=torch.float64, device=DEV)
    ops.cross_gram(Z, zn, Zt, znt, kid, osg, Kx, n, mt)
    Kxref = O.gram(p, X, Xs, training=False)
    assert (Kx[:, :n, :ns].cpu() - Kxref).abs().max().item() < tol
    assert Kx[:, n:, :].abs().max().item() == 0.0 if np_ > n else True


@pytest.mark.parametrize("kind,kid", [("rbf", 0), ("matern52", 1), ("matern32", 2), ("matern12", 3)])
@pytest.mark.parametrize("n,d,with_os", [(100, 1, False), (300, 6, True), (257, 21, False), (640, 12, True),
                                         (200, 24, False), (150, 30, True)])
def test_gradient_sweep_both_kernels_vs_autograd(kind, kid, n, d, with_os):
    """plmc_grad_sweep against torch autograd through the oracle's kernel function, f = sum_ij W_ij K_ij with
    W = 1/2 (a a^T - Kinv) held fixed: the GEMM-form kernel (d <= 24: distances and A Z on DMMA, two CTAs per SM)
    and the direct-difference kernel (any d <= 44; forced with plmc_sweep_debug) must both match."""
    q = 2
    g = torch.Generator().manual_seed(n * 31 + d)
    X = torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1
    ell = (torch.rand(q, d, generator=g, dtype=torch.float64) + 0.4).requires_grad_(True)
    os_ = (torch.rand(q, generator=g, dtype=torch.float64) + 0.5).requires_grad_(True) if with_os else None
    a = torch.randn(q, n, generator=g, dtype=torch.float64)
    M = torch.randn(q, n, n, generator=g, dtype=torch.float64)
    Kinv = M @ M.transpose(1, 2) / n
    W = 0.5 * (a[:, :, None] * a[:, None, :] - Kinv)
    f = torch.zeros((), dtype=torch.float64)
    for l in range(q):
        Kl = O.base_kernel(kind, X, X, ell[l:l + 1], zero_diag=True)
        if os_ is not None:
            Kl = os_[l] * Kl
        f = f + (W[l] * Kl).sum()
    f.backward()
    np_ = ops.npad(n)
    Xg = X.to(DEV)
    Z, zn = ops.scale_inputs(Xg, ops.col_mean(Xg), ell.detach().to(DEV), np_)
    Kp = torch.full((q, np_, np_), float("nan"), dtype=torch.float64, device=DEV)
    Kp[:, :, :] = torch.eye(np_, dtype=torch.float64, device=DEV)
    Kp[:, :n, :n] = torch.tril(Kinv).to(DEV) + torch.triu(torch.full((n, n), float("nan"), dtype=torch.float64), 1).to(DEV)
    ap = torch.zeros((q, np_), dtype=torch.float64, device=DEV)
    ap[:, :n] = a.to(DEV)
    osg = None if os_ is None else os_.detach().to(DEV)
    try:
        for direct in (False, True):
            ops.sweep_debug(direct)
            g_ell, g_os, g_noise = ops.grad_sweep(Kp, ap, Z, zn, ell.detach().to(DEV), kid, osg, n)
            assert rel_err(g_ell, ell.grad) < 1e-10, (direct, g_ell.cpu(), ell.grad)
            assert rel_err(g_noise, torch.diagonal(W, dim1=1, dim2=2).sum(-1)) < 1e-12, direct
            if os_ is not None:
                assert rel_err(g_os, os_.grad) < 1e-11, direct
    finally:
        ops.sweep_debug(False)


def test_prediction_epilogues():
    q, n, ns, p = 5, 300, 200, 37
    np_, mt = ops.npad(n), ops.npad(ns)
    Kx = rnd(q, np_, mt, seed=1)
    Kx[:, n:, :] = 0
    alpha = rnd(q, n, seed=2)
    lm = ops.latent_mean(Kx, alpha, n, mt)
    assert (lm[:, :ns] - torch.einsum("qi,qij->qj", alpha, Kx[:, :n, :ns])).abs().max().item() < 1e-11
    os_ = torch.rand(q, dtype=torch.float64, device=DEV) + 0.5
    lv = ops.latent_var(Kx, os_, mt)
    assert (lv[:, :ns] - (os_[:, None] - Kx[:, :, :ns].pow(2).sum(1))).abs().max().item() < 1e-10
    H = rnd(q, p, seed=3)
    va = torch.rand(p, dtype=torch.float64, device=DEV)
    mean = torch.empty(ns, p, dtype=torch.float64, device=DEV)
    var = torch.empty_like(mean)
    ops.mix_tasks(lm, lv, H, va, mean, var, ns)
    assert (mean - lm[:, :ns].T @ H).abs().max().item() < 1e-11
    assert (var - (lv[:, :ns].T @ H.pow(2) + va)).abs().max().item() < 1e-10
    ops.mix_tasks(lm, lv, H, va, mean, var, ns, accumulate=True)
    assert (mean - 2 * lm[:, :ns].T @ H).abs().max().item() < 1e-11


def test_large_n_properties():
    """n = 8192 (beyond a quick CPU oracle): residual, symmetry and determinant properties."""
    n, q, d = 8192, 2, 5
    g = torch.Generator().manual_seed(0)
    X = (torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1).to(DEV)
    ell = torch.full((q, d), 0.7, dtype=torch.float64, device=DEV)
    noise = torch.tensor([0.3, 0.05], dtype=torch.float64, device=DEV)
    Z, zn = ops.scale_inputs(X, ops.col_mean(X), ell, n)
    K = torch.empty((q, n, n), dtype=torch.float64, device=DEV)
    ops.gram(Z, zn, 1, None, noise, K, n)
    Kfull = torch.tril(K) + torch.tril(K, -1).transpose(1, 2)
    dinv = ops.alloc_dinv(n, q, DEV)
    info = torch.zeros(q, dtype=torch.int32, device=DEV)
    ops.potrf(K, dinv, info)
    assert info.tolist() == [0, 0]
    y = rnd(q, n, seed=4)
    z, alpha, quad, logdet = ops.solve_logdet(K, dinv, y, n)
    resid = (Kfull @ alpha.unsqueeze(-1)).squeeze(-1) - y
    assert resid.abs().max().item() < 1e-9 * y.abs().max().item() * 10
    assert torch.allclose(quad, (alpha * y).sum(-1), rtol=1e-10)              # y^T K^-1 y two ways
    assert torch.allclose(logdet, torch.linalg.slogdet(Kfull)[1], rtol=1e-10)
    ops.potri(K, dinv)
    Kinv = torch.tril(K) + torch.tril(K, -1).transpose(1, 2)
    v = rnd(q, n, 3, seed=5)
    assert ((Kfull @ (Kinv @ v)) - v).abs().max().item() < 1e-8               # K K^-1 v = v
