"""GPU: the Gram / cross-Gram, gradient-sweep and SGPR-adjoint kernels against the float64 direct-difference
reference (tests/kernel_reference.py) on every staging, tiling and reduction path:

* Gram and cross-Gram: d in {1, 21, 24} (one staged chunk), 25 (dpad 28, chunk width kcmax = 32), 33 and 44 (two
  chunks with a ragged last one, 32 + 4 and 32 + 12); n from 1 to 4500 (666 lower tiles); ld > npad; the
  additive (``accumulate``) form; the exp flush.  Every entry is held to the reference's entry-wise bound.
* Gradient sweep: the GEMM form (d <= 24, NB = 1, 2, 3), the direct form (d = 25, 44 and forced for d <= 24), and
  n = 4500 / 6000, where CTAs of the 592-CTA grid walk two tiles.
* SGPR adjoint: 1-3 row tiles, 1-3 column chunks, 1-3 passes of SG_DC = 16 dimensions, a strided cotangent, and
  autograd through ``sgpr.CrossGram``.

Gradients are held to ``prop + C_GRAD u abs`` (kernel_reference's module docstring): C_GRAD = 2^12 covers the longest
sequential chain of additions behind one device sum (an SGPR row-gradient thread adds up to 2048 columns of its
chunk half; the sweep reduces 592 CTA partials in order) plus the few ulp of each term."""
import math

import numpy as np
import pytest
import torch

from projected_lmc_b200 import ops, sgpr

from . import kernel_reference as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = R.U
C_GRAD = 4096
SENTINEL = -12345.678
TINY = 2.2250738585072014e-308      # smallest normal double
ALPHAS = np.array([0.05, 1.0, 1e4])  # RQ: distinct alpha per latent


def _data(n, d, q, seed, with_os=True, kid=0):
    """Inputs with an exact duplicate row (off-diagonal s = 0) and a zero-variance column; lengthscales ~ sqrt(d)
    so that kernel values span (0, 1) at every d.  The zero-variance column is the first one: in the last column it
    would leave the last staged chunk at d = 33 (dimension 32 and three padding dimensions) all zero, and a kernel
    that skipped or truncated that chunk would go unnoticed."""
    g = np.random.default_rng(seed)
    X = g.uniform(-1.0, 1.0, (n, d))
    if n > 2:
        X[n - 1] = X[1]
    if d > 1:
        X[:, 0] = 0.375
    ell = g.uniform(0.3, 0.9, (q, d)) * math.sqrt(d)
    os_ = g.uniform(0.5, 1.5, q) if with_os else None
    alpha = np.resize(ALPHAS if q == 3 else np.roll(ALPHAS, seed), q) if kid == 4 else None
    return X, ell, os_, alpha, g


def _dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _scaled(X, xm, ell, rows_pad):
    Z, zn = ops.scale_inputs(_dev(X), xm, _dev(ell), rows_pad)
    z = R.scale(X, xm.cpu().numpy(), ell)
    d = X.shape[1]
    # same xbar: the device's scaled inputs are the reference's, bit for bit
    assert torch.equal(Z[:, :X.shape[0], :d].cpu(), torch.from_numpy(z))
    return Z, zn, z


def _ref_entries(kid, zr, zc, os_, alpha, dpad):
    """Per latent: reference values, bound, must-flush and may-flush masks (expansion-form distances)."""
    out = []
    for l in range(zr.shape[0]):
        s = R.sq_dist(zr[l], zc[l])
        ds = R.ds_bound(s, (zr[l] ** 2).sum(1), (zc[l] ** 2).sum(1), dpad)
        o = 1.0 if os_ is None else os_[l]
        a = None if alpha is None else alpha[l]
        bound, must, may = R.entry_bound(kid, s, ds, o, a)
        out.append((o * R.profile(kid, s, a)[0], bound, must, may))
    return out


def _check_entries(got, ref, bound, must, may, what):
    assert np.isfinite(got).all(), what
    assert not ((got != 0) & (np.abs(got) < TINY)).any(), f"{what}: denormal"
    assert (got[must] == 0.0).all(), f"{what}: an entry past the exp flush is not 0"
    ok = (np.abs(got - ref) <= bound) | (may & (got == 0.0))
    if not ok.all():
        i = np.unravel_index(np.argmax(np.where(ok, 0, np.abs(got - ref) / np.maximum(bound, 1e-300))), got.shape)
        pytest.fail(f"{what}: {(~ok).sum()} entries out of bound, e.g. {i}: got {got[i]!r} ref {ref[i]!r} "
                    f"bound {bound[i]!r}")


def _run_gram(kid, X, ell, os_, alpha, noise, Xs=None, xm=None):
    """Gram into a [q, npad, npad + 6] buffer (ld > npad) and, with Xs, the cross-Gram into [q, npad, mt + 2]."""
    n, d = X.shape
    q = ell.shape[0]
    np_ = ops.npad(n)
    Xg = _dev(X)
    xm = ops.col_mean(Xg) if xm is None else xm
    Z, zn, z = _scaled(X, xm, ell, np_)
    buf = torch.full((q, np_, np_ + 6), SENTINEL, dtype=torch.float64, device=DEV)
    ops.gram(Z, zn, kid, _dev(os_), _dev(noise), buf[:, :, :np_], n, shape=_dev(alpha))
    out = {"K": buf.cpu().numpy(), "z": z, "np": np_, "xm": xm, "Z": Z, "zn": zn}
    if Xs is not None:
        mt = ops.npad(Xs.shape[0])
        Zt, znt, zt = _scaled(Xs, xm, ell, mt)
        xbuf = torch.full((q, np_, mt + 2), SENTINEL, dtype=torch.float64, device=DEV)
        ops.cross_gram(Z, zn, Zt, znt, kid, _dev(os_), xbuf[:, :, :mt], n, mt, shape=_dev(alpha))
        out.update(Kx=xbuf.cpu().numpy(), zt=zt, mt=mt)
    return out


def _check_gram_layout(K, n, np_):
    """Identity padding in the lower tiles, sentinels in the strictly upper 128-tiles and the ld - npad slack."""
    q = K.shape[0]
    assert (K[:, :, np_:] == SENTINEL).all(), "ld - npad slack columns written"   # (none when ld = npad)
    t = np.arange(np_) // 128
    upper = t[:, None] < t[None, :]
    assert (K[:, :, :np_][:, upper] == SENTINEL).all(), "strictly upper tile written"
    lower = ~upper
    pad = np.zeros((np_, np_), dtype=bool)
    pad[n:, :] = True
    pad[:, n:] = True
    sel = pad & lower
    eye = np.broadcast_to(np.eye(np_), (q, np_, np_))
    assert np.array_equal(K[:, :, :np_][:, sel], eye[:, sel]), "padding is not the identity"


def _check_gram_values(kid, res, os_, alpha, noise, dpad):
    K, z, np_ = res["K"], res["z"], res["np"]
    n = z.shape[1]
    t = np.arange(n) // 128
    low = t[:, None] >= t[None, :]          # every entry the kernel writes inside n x n
    for l, (ref, bound, must, may) in enumerate(_ref_entries(kid, z, z, os_, alpha, dpad)):
        ref = ref.copy()
        ref[np.diag_indices(n)] += noise[l]
        bound = bound + 2 * U * np.abs(ref)
        got = K[l, :n, :n]
        _check_entries(np.where(low, got, 0.0), np.where(low, ref, 0.0), bound, must & low, may, f"K[{l}]")


def _check_cross_values(kid, res, os_, alpha, dpad, ns):
    Kx, z, zt = res["Kx"], res["z"], res["zt"]
    n, mt = z.shape[1], res["mt"]
    assert (Kx[:, :, mt:] == SENTINEL).all(), "ldx - mt slack columns written"
    assert (Kx[:, n:, :mt] == 0.0).all(), "padded cross-Gram rows are not 0"
    for l, (ref, bound, must, may) in enumerate(_ref_entries(kid, z, zt, os_, alpha, dpad)):
        _check_entries(Kx[l, :n, :ns], ref, bound, must, may, f"Kx[{l}]")


GRAM_CASES = [  # kid, d, n, q, with_os
    (0, 1, 1, 3, True), (1, 21, 127, 3, False), (2, 24, 128, 1, True), (3, 25, 129, 3, True),
    (4, 28, 257, 3, False), (0, 33, 257, 3, True), (1, 44, 129, 3, True), (4, 44, 128, 3, True),
    (3, 33, 127, 1, False), (2, 28, 1, 3, False), (2, 44, 257, 3, True), (3, 1, 257, 3, False),
    (4, 1, 129, 3, True), (0, 24, 129, 1, False), (1, 28, 257, 1, True),
    (4, 44, 4500, 1, True), (3, 25, 4500, 1, False),
]


@pytest.mark.parametrize("kid,d,n,q,with_os", GRAM_CASES)
def test_gram_and_cross_gram_vs_reference(kid, d, n, q, with_os):
    X, ell, os_, alpha, g = _data(n, d, q, seed=1000 * kid + 10 * d + n % 7, with_os=with_os, kid=kid)
    noise = g.uniform(0.01, 0.3, q)
    ns = 300                                           # three column tiles, the last one ragged
    Xs = g.uniform(-1.2, 1.2, (ns, d))
    Xs[5] = X[0]                                       # a test point on a training point
    res = _run_gram(kid, X, ell, os_, alpha, noise, Xs)
    dpad = ops.dpad_of(d)
    _check_gram_layout(res["K"], n, res["np"])
    _check_gram_values(kid, res, os_, alpha, noise, dpad)
    _check_cross_values(kid, res, os_, alpha, dpad, ns)


@pytest.mark.parametrize("kid", [0, 1, 2, 3, 4])
def test_gram_flushes_to_zero_past_the_exp_range(kid):
    """Points on a line whose pair distances take the exp argument from 0 to about -1400: the entries past -707 are
    exactly 0 (no NaN, no denormal), those just inside it meet the relative bound."""
    n, d, q = 129, 2, 1
    g = np.random.default_rng(kid)
    top = {0: 2 * 1400.0, 1: (1400.0 / math.sqrt(5)) ** 2, 2: (1400.0 / math.sqrt(3)) ** 2, 3: 1400.0 ** 2}
    alpha = np.array([1e4]) if kid == 4 else None
    s_max = 2 * 1e4 * math.expm1(1400.0 / 1e4) if kid == 4 else top[kid]
    X = np.zeros((n, d))
    X[:, 0] = np.arange(n) * (math.sqrt(s_max) / (n - 1))
    X[:, 1] = g.uniform(-0.1, 0.1, n)
    ell = np.ones((q, d))
    noise = np.array([0.1])
    res = _run_gram(kid, X, ell, None, alpha, noise, Xs=X[::-1].copy())
    z = res["z"][0]
    arg = R.profile(kid, R.sq_dist(z, z), None if alpha is None else alpha[0])[3]
    assert (arg < -712).sum() > 100 and ((arg > -707) & (arg < -680)).sum() > 20   # both sides are exercised
    _check_gram_layout(res["K"], n, res["np"])
    _check_gram_values(kid, res, None, alpha, noise, 4)
    _check_cross_values(kid, res, None, alpha, 4, n)


def test_additive_gram_adds_noise_and_padding_once():
    """Matern-5/2 on dims 0-9 plus RQ on dims 10-32 (dpad 12, then 24), the second with accumulate = 1, in the Gram
    and the cross-Gram: the noise and the identity padding are written once, the components add."""
    n, ns, q = 257, 200, 3
    X, _, _, _, g = _data(n, 33, q, seed=5)
    Xs = g.uniform(-1, 1, (ns, 33))
    comps = [(1, list(range(0, 10)), g.uniform(0.5, 1.5, q), None),
             (4, list(range(10, 33)), g.uniform(0.5, 1.5, q), ALPHAS)]
    noise = g.uniform(0.05, 0.2, q)
    np_, mt = ops.npad(n), ops.npad(ns)
    K = torch.full((q, np_, np_), SENTINEL, dtype=torch.float64, device=DEV)
    Kx = torch.full((q, np_, mt), SENTINEL, dtype=torch.float64, device=DEV)
    ref, bound = np.zeros((q, n, n)), np.zeros((q, n, n))
    refx, boundx = np.zeros((q, n, ns)), np.zeros((q, n, ns))
    for c, (kid, dims, os_, alpha) in enumerate(comps):
        Xc, Xsc = np.ascontiguousarray(X[:, dims]), np.ascontiguousarray(Xs[:, dims])
        ell = g.uniform(0.3, 0.9, (q, len(dims))) * math.sqrt(len(dims))
        xm = ops.col_mean(_dev(Xc))
        Z, zn, z = _scaled(Xc, xm, ell, np_)
        Zt, znt, zt = _scaled(Xsc, xm, ell, mt)
        ops.gram(Z, zn, kid, _dev(os_), _dev(noise), K, n, accumulate=c > 0, shape=_dev(alpha))
        ops.cross_gram(Z, zn, Zt, znt, kid, _dev(os_), Kx, n, mt, accumulate=c > 0, shape=_dev(alpha))
        dp = ops.dpad_of(len(dims))
        for l, (r, b, _, may) in enumerate(_ref_entries(kid, z, z, os_, alpha, dp)):
            ref[l] += r
            bound[l] += b + np.where(may, np.abs(r), 0.0)
        for l, (r, b, _, may) in enumerate(_ref_entries(kid, z, zt, os_, alpha, dp)):
            refx[l] += r
            boundx[l] += b + np.where(may, np.abs(r), 0.0)
    ref[:, np.arange(n), np.arange(n)] += noise[:, None]
    Kc, Kxc = K.cpu().numpy(), Kx.cpu().numpy()
    _check_gram_layout(Kc, n, np_)
    t = np.arange(n) // 128
    low = t[:, None] >= t[None, :]
    none, nonex = np.zeros((n, n), dtype=bool), np.zeros((n, ns), dtype=bool)
    for l in range(q):   # + the rounding of the sum of the two components and the noise
        _check_entries(np.where(low, Kc[l, :n, :n], 0), np.where(low, ref[l], 0), bound[l] + 4 * U * np.abs(ref[l]),
                       none, none, f"K[{l}]")
        _check_entries(Kxc[l, :n, :ns], refx[l], boundx[l] + 4 * U * np.abs(refx[l]), nonex, nonex, f"Kx[{l}]")
    assert (Kxc[:, n:, :] == 0.0).all()


def test_col_mean_at_n_100003_against_fsum():
    n, d = 100003, 3
    X = 1e3 + np.random.default_rng(3).uniform(-1, 1, (n, d))
    got = ops.col_mean(_dev(X)).cpu().numpy()
    ref = R.col_mean(X)
    # 256 threads each add about n / 256 values in order, then a tree over the block: (n / 256 + 16) u max|x|
    assert (np.abs(got - ref) <= (n / 256 + 16) * U * np.abs(X).max()).all(), got - ref


# ---------------------------------------------------------------------------------------------------------------
# gradient sweep
# ---------------------------------------------------------------------------------------------------------------
SWEEP_CASES = [  # kid, d, n, q, with_os, form ("gemm": d <= 24 default, "direct": d > 24, "forced": sweep_debug)
    (0, 2, 129, 3, True, "gemm"), (1, 12, 129, 3, False, "gemm"), (2, 24, 129, 3, True, "gemm"),
    (3, 12, 129, 3, True, "gemm"), (4, 24, 129, 3, True, "gemm"), (3, 2, 129, 3, False, "gemm"),
    (0, 25, 129, 3, False, "direct"), (1, 44, 129, 3, True, "direct"), (2, 44, 129, 3, False, "direct"),
    (3, 25, 129, 3, True, "direct"), (4, 44, 129, 3, True, "direct"),
    (4, 12, 129, 3, True, "forced"), (3, 2, 129, 3, True, "forced"), (2, 24, 129, 3, False, "forced"),
    (3, 12, 4500, 1, True, "gemm"), (4, 44, 4500, 1, True, "direct"),
    (1, 24, 6000, 1, False, "gemm"), (2, 25, 6000, 1, True, "direct"),
]


def _sweep_inputs(kid, d, n, q, with_os):
    """alpha on a 2^-8 grid and K^-1 on a 2^-16 grid (symmetric, indefinite), so that W = (alpha alpha^T - K^-1) / 2
    is exact in float64 however the kernel forms it; W has mixed signs."""
    X, ell, os_, alpha, g = _data(n, d, q, seed=7 * n + d + kid, with_os=with_os, kid=kid)
    a = np.round(g.standard_normal((q, n)) * 256) / 256
    Kinv = np.empty((q, n, n))
    for l in range(q):
        M = np.round(g.standard_normal((n, n)) * (65536 / math.sqrt(n))) / 65536
        Kinv[l] = M + M.T
    W = 0.5 * (a[:, :, None] * a[:, None, :] - Kinv)
    return X, ell, os_, alpha, a, Kinv, W


def _run_sweep(kid, X, ell, os_, alpha, a, Kinv):
    """K^-1 in a [q, npad, npad + 2] buffer (ld > npad) with NaN in its strict upper part and its padding, alpha
    with lda_vec = n + 5 > n and NaN past n.  Returns (the outputs as numpy, the call's arguments, z)."""
    n, d = X.shape
    q = ell.shape[0]
    np_ = ops.npad(n)
    Z, zn, z = _scaled(X, ops.col_mean(_dev(X)), ell, np_)
    Kp = torch.full((q, np_, np_ + 2), float("nan"), dtype=torch.float64, device=DEV)
    nan_up = torch.triu(torch.full((n, n), float("nan"), dtype=torch.float64, device=DEV), 1)
    for l in range(q):
        Kp[l, :n, :n] = torch.from_numpy(np.tril(Kinv[l])).to(DEV) + nan_up
    abuf = torch.full((q, n + 5), float("nan"), dtype=torch.float64, device=DEV)
    abuf[:, :n] = _dev(a)
    args = (Kp[:, :, :np_], abuf[:, :n], Z, zn, _dev(ell), kid, _dev(os_), n)
    return [t.cpu().numpy() for t in ops.grad_sweep(*args, shape=_dev(alpha))], args, z


def _check_grad(got, ref, name, C=C_GRAD):
    err = np.abs(got - ref[name])
    tol = ref[name + "_prop"] + C * U * ref[name + "_abs"]
    assert (err <= tol).all(), f"{name}: err {err} tol {tol} got {got} ref {ref[name]}"


@pytest.mark.parametrize("kid,d,n,q,with_os,form", SWEEP_CASES)
def test_gradient_sweep_vs_reference(kid, d, n, q, with_os, form):
    """Every case has an exact duplicate row.  The direct forms see s = 0 there exactly (dk/ds = 0 for nu = 1/2) and
    their tolerance stays near 1e-10 of |g_ell| for every kernel.

    Matern-1/2 in GEMM form differs in semantics, not by a defect: the GEMM form evaluates sum_ij A_ij (z_ik - z_jk)^2
    by expansion, so a pair at distance r contributes dk/ds ~ -k / (2 r) times an expanded square that carries a
    rounding error of ~u |z|^2 rather than ~u r^2, and at the duplicate it sees s ~ u |z|^2 (about 1e-15) instead of
    0, so dk/ds ~ -1e7 where the direct form takes 0.  The reference's tolerance follows this through dk/ds over the
    interval of s (``prop`` + C_GRAD u ``abs``): for these cases it comes to a median of ~7e-5 and a maximum of
    ~1.4e-2 of |g_ell| (d = 12, n = 129; ~2e-3 without the duplicate), against a median of ~1e-10 for the other
    kernels and forms (at most ~4e-6, for a g_ell that nearly cancels).  The last assertion keeps both at that size."""
    X, ell, os_, alpha, a, Kinv, W = _sweep_inputs(kid, d, n, q, with_os)
    try:
        ops.sweep_debug(form == "forced")
        out, args, z = _run_sweep(kid, X, ell, os_, alpha, a, Kinv)
        again = [t.cpu().numpy() for t in ops.grad_sweep(*args, shape=_dev(alpha))]
    finally:
        ops.sweep_debug(False)
    for x, y in zip(out, again):
        assert np.array_equal(x, y), "two calls differ"
    ref = R.sweep(kid, z, W, ell, os_, alpha, ops.dpad_of(d), expansion=form == "gemm")
    g_ell, g_os, g_noise = out[:3]
    _check_grad(g_ell, ref, "g_ell")
    _check_grad(g_os, ref, "g_os")
    _check_grad(g_noise, ref, "g_noise")          # g_noise = tr W
    if kid == 4:
        _check_grad(out[3], ref, "g_shape")
    rel = ((ref["g_ell_prop"] + C_GRAD * U * ref["g_ell_abs"]) / np.abs(ref["g_ell"]))[:, 1:]   # column 0: constant
    assert rel.max() < (2e-2 if (kid == 3 and form == "gemm") else 1e-4), rel.max()


# ---------------------------------------------------------------------------------------------------------------
# SGPR cross-Gram adjoint
# ---------------------------------------------------------------------------------------------------------------
BWD_CASES = [  # kid, nr, nc, d, q, with_os: nr 40/128/300 -> 1/1/3 row tiles; nc 330/4097/9000 -> 1/2/3 column
    # chunks; d 3/16/17/33/44 -> 1/1/2/3/3 passes of SG_DC = 16
    (0, 40, 330, 3, 3, True), (1, 128, 4097, 16, 1, False), (2, 300, 9000, 17, 1, True),
    (3, 300, 330, 33, 3, False), (4, 40, 9000, 44, 3, True), (4, 128, 330, 17, 3, False),
    (0, 300, 4097, 44, 1, True), (1, 40, 4097, 33, 3, True), (3, 128, 9000, 3, 1, True),
    (2, 40, 330, 16, 3, False), (3, 300, 4097, 17, 3, True), (4, 300, 330, 3, 1, True),
]


def _bwd_inputs(kid, nr, nc, d, q, with_os):
    X, ell, os_, alpha, g = _data(nc, d, q, seed=3 * nc + nr + d + kid, with_os=with_os, kid=kid)
    Uin = g.uniform(-1.0, 1.0, (nr, d))
    Uin[: min(nr, 7)] = X[: min(nr, 7)]                # inducing points on training points: s = 0
    return X, Uin, ell, os_, alpha, g


@pytest.mark.parametrize("kid,nr,nc,d,q,with_os", BWD_CASES)
def test_cross_gram_bwd_vs_reference(kid, nr, nc, d, q, with_os):
    X, Uin, ell, os_, alpha, g = _bwd_inputs(kid, nr, nc, d, q, with_os)
    xm = ops.col_mean(_dev(X))
    Zr, _, zr = _scaled(Uin, xm, ell, ops.npad(nr))
    Zc, _, zc = _scaled(X, xm, ell, ops.npad(nc))
    G = g.standard_normal((q, nr, nc))
    gbuf = torch.full((q, nr + 3, nc + 5), float("nan"), dtype=torch.float64, device=DEV)   # ldg > nc,
    gbuf[:, :nr, :nc] = _dev(G)                                                             # strideG > nr ldg
    Gd = gbuf[:, :nr, :nc]
    args = (Zr, Zc, Gd, kid, _dev(os_), _dev(ell), nr, nc)
    out = [t.cpu().numpy() for t in ops.cross_gram_bwd(*args, shape=_dev(alpha))]
    again = [t.cpu().numpy() for t in ops.cross_gram_bwd(*args, shape=_dev(alpha))]
    for x, y in zip(out, again):
        assert np.array_equal(x, y), "two calls differ"
    ref = R.cross_gram_bwd(kid, zr, zc, G, ell, os_, alpha)
    for name, v in zip(("g_ell", "g_os", "g_rows", "g_shape"), out):
        _check_grad(v, ref, name)


@pytest.mark.parametrize("kid", [0, 1, 2, 3, 4])
def test_sgpr_cross_gram_autograd_vs_reference(kid):
    """sgpr.CrossGram forward and backward for K_uu (symmetric: G + G^T for the points, halved lengthscale,
    outputscale and shape sums) and K_uf, with inducing points that coincide with training points (s = 0 on the
    diagonal of K_uu and at the coinciding pairs: nu = 1/2 has dk/ds = 0 there)."""
    m, n, d, q = 300, 700, 17, 3
    X, Uin, ell, os_, alpha, g = _bwd_inputs(kid, m, n, d, q, True)
    Uin[100:140] = X[200:240]
    xm = ops.col_mean(_dev(X))
    Ut = _dev(Uin).requires_grad_(True)
    ell_t = _dev(ell).requires_grad_(True)
    os_t = _dev(os_).requires_grad_(True)
    al_t = None if alpha is None else _dev(alpha).requires_grad_(True)
    Kuu = sgpr.CrossGram.apply(Ut, Ut, xm, kid, ell_t, os_t, True, al_t)
    Kuf = sgpr.CrossGram.apply(Ut, _dev(X), xm, kid, ell_t, os_t, False, al_t)
    Guu, Guf = g.standard_normal((q, m, m)), g.standard_normal((q, m, n))
    ((Kuu * _dev(Guu)).sum() + (Kuf * _dev(Guf)).sum()).backward()

    xmn = xm.cpu().numpy()
    zu, zx = R.scale(Uin, xmn, ell), R.scale(X, xmn, ell)
    dpad = ops.dpad_of(d)
    for got, zc in ((Kuu, zu), (Kuf, zx)):
        gotn = got.detach().cpu().numpy()
        for l, (r, b, must, may) in enumerate(_ref_entries(kid, zu, zc, os_, alpha, dpad)):
            _check_entries(gotn[l], r, b, must, may, f"K[{l}]")
    ruu = R.cross_gram_bwd(kid, zu, zu, Guu, ell, os_, alpha)
    ruuT = R.cross_gram_bwd(kid, zu, zu, Guu.transpose(0, 2, 1).copy(), ell, os_, alpha)
    ruf = R.cross_gram_bwd(kid, zu, zx, Guf, ell, os_, alpha)
    tot = {k: ruu[k] + ruf[k] for k in ruu}
    for k in ("g_rows", "g_rows_abs", "g_rows_prop"):
        tot[k] = tot[k] + ruuT[k]
    # K_uu's adjoint runs on G + G^T and is halved: one more rounding of the 2x sums
    _check_grad(Ut.grad.cpu().numpy(), tot, "g_rows")
    _check_grad(ell_t.grad.cpu().numpy(), tot, "g_ell")
    _check_grad(os_t.grad.cpu().numpy(), tot, "g_os")
    if kid == 4:
        _check_grad(al_t.grad.cpu().numpy(), tot, "g_shape")
