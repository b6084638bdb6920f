"""CPU checks of the float64 kernel reference (tests/kernel_reference.py): against the oracle's expansion-form
kernels within the reference's own error bound, against scikit-learn's kernels, and its analytic gradients against
torch autograd and central differences."""
import math

import numpy as np
import pytest
import torch

from oracle import plmc_oracle as O

from . import kernel_reference as R
from .rq_reference import rq_kernel

KINDS = {0: "rbf", 1: "matern52", 2: "matern32", 3: "matern12"}


def _inputs(n, d, seed, q=2):
    g = np.random.default_rng(seed)
    X = g.uniform(-1.0, 1.0, (n, d))
    ell = g.uniform(0.4, 1.4, (q, d))
    return X, ell, g


@pytest.mark.parametrize("kid", [0, 1, 2, 3, 4])
def test_reference_gram_matches_oracle_within_the_bound(kid):
    n, d, q = 70, 5, 2
    X, ell, g = _inputs(n, d, kid)
    X[7] = X[3]                                   # a duplicate row: off-diagonal s = 0
    os_ = g.uniform(0.5, 1.5, q)
    alpha = np.array([0.3, 7.0])
    noise = np.array([0.1, 0.02])
    z = R.scale(X, R.col_mean(X), ell)
    K = R.gram(kid, z, os_, alpha if kid == 4 else None, noise)
    Xt, ellt = torch.from_numpy(X), torch.from_numpy(ell)[:, None, :]
    if kid == 4:
        Ko = rq_kernel(Xt, Xt, ellt, True, torch.from_numpy(alpha)[:, None]).numpy()
    else:
        Ko = O.base_kernel(KINDS[kid], Xt, Xt, ellt, zero_diag=True).numpy()
    Ko = Ko * os_[:, None, None] + noise[:, None, None] * np.eye(n)
    for l in range(q):
        nz = (z[l] ** 2).sum(1)
        s = R.sq_dist(z[l], z[l])
        bound = R.entry_bound(kid, s, R.ds_bound(s, nz, nz, 8), os_[l], alpha[l] if kid == 4 else None)[0]
        bound += 2 * R.U * np.abs(K[l])          # the noise addition
        assert (np.abs(K[l] - Ko[l]) <= bound).all(), np.abs(K[l] - Ko[l]).max()


@pytest.mark.parametrize("kid,nu,alpha", [(0, None, None), (3, 0.5, None), (2, 1.5, None), (1, 2.5, None),
                                          (4, None, 0.05), (4, None, 1.0), (4, None, 1e4)])
def test_reference_matches_scikit_learn(kid, nu, alpha):
    from sklearn.gaussian_process.kernels import RBF, Matern, RationalQuadratic

    X, ell, g = _inputs(40, 3, 11, q=1)
    X2 = g.uniform(-1.5, 1.5, (25, 3))
    X2[4] = X[9]                                  # s = 0 in the cross block
    z1, z2 = R.scale(X, np.zeros(3), ell), R.scale(X2, np.zeros(3), ell)
    K = R.cross_gram(kid, z1, z2, alpha=None if alpha is None else np.array([alpha]))[0]
    if kid == 0:
        sk = RBF(length_scale=1.0)
    elif kid == 4:
        sk = RationalQuadratic(length_scale=1.0, alpha=alpha)
    else:
        sk = Matern(length_scale=1.0, nu=nu)
    ref = sk(z1[0], z2[0])                       # ARD by pre-scaling the inputs
    s = R.sq_dist(z1[0], z2[0])
    bound = R.entry_bound(kid, s, R.ds_bound(s, None, None, 4, expansion=False), 1.0, alpha)[0]
    # scikit-learn evaluates RQ as (1 + s / 2 alpha) ** -alpha: rounding 1 + s / 2 alpha costs it alpha u relative
    slack = (4 + (2 * alpha if kid == 4 else 0)) * R.U * np.abs(ref)
    assert (np.abs(K - ref) <= bound + slack).all(), np.abs(K - ref).max()


def test_flush_region_and_bound_conventions():
    # the exp argument past -707 is flagged as a flush for every kernel; just inside it is not
    for kid, s_in, s_out in ((0, 1412.0, 1416.0), (1, (706.0 / math.sqrt(5)) ** 2, (708.0 / math.sqrt(5)) ** 2),
                             (3, 706.0 ** 2, 708.0 ** 2)):
        s = np.array([[s_in, s_out]])
        _, must, may = R.entry_bound(kid, s, np.zeros_like(s))
        assert must.tolist() == [[False, True]] and may.tolist() == [[False, True]]
    # nu = 1/2: dk/ds = 0 at s <= 1e-30 and the bound at s = 0 is sqrt(ds) (not the unbounded first-order term)
    k, dk, _, _ = R.profile(3, np.array([0.0, 1e-31, 1e-20]))
    assert dk[0] == 0.0 and dk[1] == 0.0 and dk[2] < -1e9
    b = R.entry_bound(3, np.array([0.0]), np.array([1e-16]))[0]
    assert abs(b[0] - 1e-8) < 1e-10


def _t_kernel(kid, s, alpha):
    if kid == 0:
        return torch.exp(-0.5 * s)
    if kid == 4:
        return torch.exp(-alpha * torch.log1p(s / (2 * alpha)))
    a = R._RATE[kid] * s.clamp_min(1e-30).sqrt()
    e = torch.exp(-a)
    return {1: (1 + a + a * a / 3) * e, 2: (1 + a) * e, 3: e}[kid]


def _t_sq(z1, z2):
    return (z1[:, :, None, :] - z2[:, None, :, :]).pow(2).sum(-1)


@pytest.mark.parametrize("kid", [0, 1, 2, 3, 4])
def test_sweep_reference_matches_autograd_and_central_differences(kid):
    n, d, q = 33, 3, 2
    X, ell, g = _inputs(n, d, 20 + kid, q)
    xm = R.col_mean(X)
    os_ = g.uniform(0.5, 1.5, q)
    alpha = np.array([0.4, 25.0]) if kid == 4 else None
    A = g.standard_normal((q, n, n))
    a = g.standard_normal((q, n))
    W = 0.5 * (a[:, :, None] * a[:, None, :] - (A + A.transpose(0, 2, 1)))
    ref = R.sweep(kid, R.scale(X, xm, ell), W, ell, os_, alpha, expansion=False)

    ell_t = torch.tensor(ell, requires_grad=True)
    os_t = torch.tensor(os_, requires_grad=True)
    al_t = torch.tensor(alpha if kid == 4 else np.ones(q), requires_grad=True)
    noise_t = torch.zeros(q, requires_grad=True)
    z = (torch.from_numpy(X) - torch.from_numpy(xm))[None] / ell_t[:, None, :]
    K = os_t[:, None, None] * _t_kernel(kid, _t_sq(z, z), al_t[:, None, None]) + noise_t[:, None, None] * torch.eye(n)
    (torch.from_numpy(W) * K).sum().backward()
    C = 64 * R.U
    for name, t in (("g_ell", ell_t), ("g_os", os_t), ("g_noise", noise_t)):
        assert (np.abs(ref[name] - t.grad.numpy()) <= C * ref[name + "_abs"]).all(), name
    if kid == 4:
        assert (np.abs(ref["g_shape"] - al_t.grad.numpy()) <= C * ref["g_shape_abs"]).all()

    # central differences of f = sum W K through the reference Gram
    def f(ell_, alpha_):
        return sum(math.fsum((W[l] * R.gram(kid, R.scale(X, xm, ell_), os_, alpha_)[l]).ravel()) for l in range(q))

    h = 1e-5
    for l, k in ((0, 0), (1, 2)):
        e1, e2 = ell.copy(), ell.copy()
        e1[l, k] *= 1 + h
        e2[l, k] *= 1 - h
        fd = (f(e1, alpha) - f(e2, alpha)) / (2 * h * ell[l, k])
        assert abs(fd - ref["g_ell"][l, k]) <= 1e-7 * ref["g_ell_abs"][l, k]
    if kid == 4:
        a1, a2 = alpha.copy(), alpha.copy()
        a1[0] *= 1 + h
        a2[0] *= 1 - h
        fd = (f(ell, a1) - f(ell, a2)) / (2 * h * alpha[0])
        assert abs(fd - ref["g_shape"][0]) <= 1e-7 * ref["g_shape_abs"][0]


@pytest.mark.parametrize("kid", [0, 1, 2, 3, 4])
def test_cross_gram_bwd_reference_matches_autograd_and_central_differences(kid):
    nr, nc, d, q = 17, 29, 4, 2
    X, ell, g = _inputs(nc, d, 40 + kid, q)
    Uin = g.uniform(-1.0, 1.0, (nr, d))
    xm = R.col_mean(X)
    os_ = g.uniform(0.5, 1.5, q)
    alpha = np.array([0.2, 3.0]) if kid == 4 else None
    G = g.standard_normal((q, nr, nc))
    ref = R.cross_gram_bwd(kid, R.scale(Uin, xm, ell), R.scale(X, xm, ell), G, ell, os_, alpha)

    u_t = torch.tensor(Uin, requires_grad=True)
    ell_t = torch.tensor(ell, requires_grad=True)
    os_t = torch.tensor(os_, requires_grad=True)
    al_t = torch.tensor(alpha if kid == 4 else np.ones(q), requires_grad=True)
    xm_t = torch.from_numpy(xm)
    zr = (u_t - xm_t)[None] / ell_t[:, None, :]
    zc = (torch.from_numpy(X) - xm_t)[None] / ell_t[:, None, :]
    K = os_t[:, None, None] * _t_kernel(kid, _t_sq(zr, zc), al_t[:, None, None])
    (torch.from_numpy(G) * K).sum().backward()
    C = 64 * R.U
    for name, t in (("g_ell", ell_t), ("g_os", os_t), ("g_rows", u_t)):
        assert (np.abs(ref[name] - t.grad.numpy()) <= C * ref[name + "_abs"]).all(), name
    if kid == 4:
        assert (np.abs(ref["g_shape"] - al_t.grad.numpy()) <= C * ref["g_shape_abs"]).all()

    def f(u_):
        Kr = R.cross_gram(kid, R.scale(u_, xm, ell), R.scale(X, xm, ell), os_, alpha)
        return math.fsum((G * Kr).ravel())

    h = 1e-6
    for i, k in ((0, 0), (5, 3), (16, 1)):
        u1, u2 = Uin.copy(), Uin.copy()
        u1[i, k] += h
        u2[i, k] -= h
        fd = (f(u1) - f(u2)) / (2 * h)
        assert abs(fd - ref["g_rows"][i, k]) <= 1e-7 * ref["g_rows_abs"][i, k]


def test_col_mean_is_correctly_rounded():
    X = np.full((3, 1), 0.1)
    X[1, 0] = 1e16
    X[2, 0] = -1e16
    assert R.col_mean(X)[0] == 0.1 / 3
