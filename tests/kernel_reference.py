"""Plain float64 CPU reference of the kernel-evaluation kernels: the Gram and cross-Gram (csrc/gram.cu
``gram_kernel``), the fused gradient sweep (``grad_sweep_kernel`` / ``grad_sweep2_kernel``) and the SGPR cross-Gram
adjoint (csrc/sgpr.cu ``cross_gram_bwd_kernel``), with the outputs of ``ops.gram``, ``ops.cross_gram``,
``ops.grad_sweep`` and ``ops.cross_gram_bwd``.  It shares no code with the oracle or the library:

* inputs are scaled as the library does, ``z = (x - xbar) / ell`` (xbar given, or ``col_mean`` by ``math.fsum``);
  with the same xbar the scaled inputs are bit-identical to the device's (one correctly rounded subtraction and
  division each);
* squared distances are summed from **direct differences**, ``s_ij = sum_k (z_ik - z_jk)^2``, in row blocks, never by
  the quadratic expansion ``|z_i|^2 + |z_j|^2 - 2 z_i.z_j`` that the device kernels and the oracle use;
* the profiles k(s), dk/ds and dk/dalpha of kernel ids 0-4 come from numpy's exp / sqrt / log1p, with the library's
  conventions: ``r = sqrt(max(s, 1e-30))``, and for nu = 1/2 ``dk/ds = 0`` at ``s <= 1e-30``.

Every gradient comes back with a scale against which a tolerance is set (``*_abs``): the sum of the absolute values
of its terms, each term taken with its largest magnitude over the interval in which the device's s can lie, and the
squared difference ``(z_ik - z_jk)^2`` replaced by ``(|z_ik| + |z_jk|)^2``, which also bounds the terms of the
expanded form ``sum_i z_ik (r_i z_ik - 2 U_ik) + sum_j c_j z_jk^2`` that the GEMM-form sweep evaluates.  Gradients
also come back with ``*_prop``: the bound of what the error of s alone (``ds_bound``) moves the result by.  A test
then accepts ``|got - ref| <= prop + C 2^-53 abs`` for a stated C, independent of cancellation in the result.
"""
import math

import numpy as np
import torch

U = 2.0 ** -53               # unit roundoff of float64
FLUSH = -707.0               # exp_nonpos returns exactly 0 below this argument
_RATE = {1: math.sqrt(5.0), 2: math.sqrt(3.0), 3: 1.0}   # Matern: sqrt(2 nu)


def col_mean(X):
    """Column means of X [n, d] by math.fsum (correctly rounded sums)."""
    X = np.asarray(X, dtype=np.float64)
    return np.array([math.fsum(X[:, k]) / X.shape[0] for k in range(X.shape[1])])


def scale(X, xmean, ell):
    """z = (x - xbar) / ell for X [n, d], xbar [d] and ell [q, d] -> [q, n, d]."""
    X, xmean, ell = (np.asarray(a, dtype=np.float64) for a in (X, xmean, ell))
    return (X[None, :, :] - xmean[None, None, :]) / ell[:, None, :]


def _blocks(n1, n2):
    """Row blocks that keep one [rows, n2] temporary near 32 MB."""
    b = max(1, (1 << 22) // max(1, n2))
    return [(i0, min(n1, i0 + b)) for i0 in range(0, n1, b)]


def sq_dist(z1, z2):
    """s_ij = sum_k (z1_ik - z2_jk)^2 by direct differences, for z1 [n1, d], z2 [n2, d]."""
    a, b = torch.from_numpy(np.ascontiguousarray(z1)), torch.from_numpy(np.ascontiguousarray(z2))
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float64)
    for i0, i1 in _blocks(a.shape[0], b.shape[0]):
        acc = out[i0:i1]
        acc.zero_()
        for k in range(a.shape[1]):
            acc.add_((a[i0:i1, k, None] - b[None, :, k]).square_())
    return out.numpy()


def profile(kid, s, alpha=None):
    """(k, dk/ds, dk/dalpha, the argument of exp) of kernel ``kid`` at squared scaled distances s (any shape).
    The argument of exp is where the library flushes: RBF -s/2, Matern -sqrt(2 nu) r, RQ -alpha log1p(s / 2 alpha)."""
    s = np.asarray(s, dtype=np.float64)
    zero = np.zeros_like(s)
    if kid == 0:
        arg = -0.5 * s
        k = np.exp(arg)
        return k, -0.5 * k, zero, arg
    if kid == 4:
        if alpha is None:
            raise ValueError("the rational quadratic kernel needs alpha")
        x = s / (2.0 * alpha)
        L = np.log1p(x)
        arg = -alpha * L
        k = np.exp(arg)
        return k, -k / (2.0 * (1.0 + x)), k * (x / (1.0 + x) - L), arg
    r = np.sqrt(np.maximum(s, 1e-30))
    a = _RATE[kid] * r
    e = np.exp(-a)
    if kid == 1:
        k, dk = (1.0 + a + a * a / 3.0) * e, -(5.0 / 6.0) * (1.0 + a) * e
    elif kid == 2:
        k, dk = (1.0 + a) * e, -1.5 * e
    else:
        k = e
        dk = np.where(s > 1e-30, -0.5 * k / r, 0.0)
    return k, dk, zero, -a


def ds_bound(s, n1, n2, dpad, expansion=True):
    """Bound of |s_device - s| for the reference's s [n1, n2] and the squared norms n1 = |z_i|^2, n2 = |z_j|^2.

    Expansion form (Gram, cross-Gram, GEMM-form sweep): the device forms |z_i|^2 by dpad FMAs and z_i.z_j by dpad
    FP64 tensor-core products, each with a relative error of at most dpad u in |z_i|^2 and in
    sum_k |z_ik z_jk| <= (|z_i|^2 + |z_j|^2) / 2, then rounds |z_i|^2 + |z_j|^2 and the final FMA
    (2 u (|z_i|^2 + |z_j|^2)).  So  ds <= (2 dpad + 4) u (|z_i|^2 + |z_j|^2).  Direct differences (the direct sweep,
    the SGPR adjoint) have a relative error of at most (dpad + 2) u in s.  The reference's own s carries the
    latter, which is added in both cases."""
    ds = (dpad + 2) * U * s
    if expansion:
        ds = ds + (2 * dpad + 4) * U * (n1[:, None] + n2[None, :])
    return ds


def entry_bound(kid, s, ds, os_=1.0, alpha=None):
    """Entry-wise bound of |K_device - os k(s)| for device distances within ds of s, and the entries that must be
    flushed.  Returns (bound, must_flush, may_flush).

    The profiles are decreasing in s and so is |dk/ds|; by the mean value theorem, with s_lo = max(s - ds, 0),
        |k(s') - k(s)| <= |dk/ds|(s_lo) ds                          for |s' - s| <= ds,
    and for nu = 1/2, whose dk/ds is unbounded at 0, |dk/dr| = k and |r' - r| <= min(ds / (2 r_lo), sqrt(ds)):
        |k(s') - k(s)| <= k(s_lo) min(ds / (2 r_lo), sqrt(ds)).
    The evaluation itself (exp to < 1 ulp, sqrt, log1p to 1.2 ulp, the polynomial factor, the outputscale product)
    adds 4 ulp(k) <= 8 u k, and the rounding of the exp argument adds its relative error (<= 6 u for RQ:
    s / 2 alpha, log1p, the product with alpha; <= 3 u for Matern) times |argument| relative to k:
        dK <= os (|dk/ds|(s_lo) ds + (8 + 8 |arg|) u k).
    Where the argument is below -707 the library flushes k to exactly 0.  The true value is then below 1e-300 (RBF
    past s = 1414; Matern past sqrt(2 nu) r = 707 with its polynomial factor; RQ past alpha log1p(s / 2 alpha) =
    707).  ``must_flush`` marks the entries whose argument is below -707 for every s' within ds (they must be
    exactly 0); ``may_flush`` those for which some s' is (0 is accepted there, or a value within the bound)."""
    s_lo = np.maximum(s - ds, 0.0)
    k, _, _, arg = profile(kid, s, alpha)
    k_lo, dk_lo, _, arg_lo = profile(kid, s_lo, alpha)
    if kid == 3:
        r_lo = np.sqrt(np.maximum(s_lo, 1e-30))
        prop = k_lo * np.minimum(ds / (2.0 * r_lo), np.sqrt(ds))
    else:
        prop = np.abs(dk_lo) * ds
    bound = os_ * (prop + (8.0 + 8.0 * np.abs(arg)) * U * k)
    arg_hi = profile(kid, s + ds, alpha)[3]
    return bound, arg_lo < FLUSH, arg_hi < FLUSH


def _shape(alpha, l):
    return None if alpha is None else float(alpha[l])


def _os(os_, l):
    return 1.0 if os_ is None else float(os_[l])


def gram(kid, z, os_=None, alpha=None, noise=None):
    """Training Gram [q, n, n] of ``ops.gram``: os k(s) plus noise[l] on the diagonal (s_ii = 0)."""
    q, n, _ = z.shape
    K = np.empty((q, n, n))
    for l in range(q):
        K[l] = _os(os_, l) * profile(kid, sq_dist(z[l], z[l]), _shape(alpha, l))[0]
        if noise is not None:
            K[l][np.diag_indices(n)] += noise[l]
    return K


def cross_gram(kid, zr, zc, os_=None, alpha=None):
    """Cross-Gram [q, nr, nc] of ``ops.cross_gram``: os k(|zr_i - zc_j|^2)."""
    return np.stack([_os(os_, l) * profile(kid, sq_dist(zr[l], zc[l]), _shape(alpha, l))[0]
                     for l in range(zr.shape[0])])


def _endpoint_delta(f, s, ds):
    """max |f(s') - f(s)| over s' in {max(s - ds, 0), s + ds}: the largest move of a monotone f within ds of s."""
    f0 = f(s)
    return np.maximum(np.abs(f(np.maximum(s - ds, 0.0)) - f0), np.abs(f(s + ds) - f0))


def _deltas(kid, s, ds, alpha):
    """Largest moves of k, dk/ds and dk/dalpha within ds of s (the last to first order: not monotone in s)."""
    return tuple(_endpoint_delta(lambda t, i=i: profile(kid, t, alpha)[i], s, ds) for i in range(3))


def _abs_scale(C, za1, za2):
    """sum_ij C_ij (|z1_ik| + |z2_jk|)^2 per k for C >= 0 [n1, n2], |z| [n1, d], [n2, d] (no cancellation)."""
    rows, cols = C.sum(1)[:, None], C.sum(0)[:, None]
    return (za1 ** 2 * rows).sum(0) + (za2 ** 2 * cols).sum(0) + 2.0 * (za1 * (C @ za2)).sum(0)


def sweep(kid, z, W, ell, os_=None, alpha=None, dpad=None, expansion=True):
    """The gradient sweep of ``ops.grad_sweep`` for f = sum_l sum_ij W_l,ij (os_l k_l(s_ij) + [i = j] sigma_l^2) with
    the full symmetric W [q, n, n] (the device reads its lower triangle and weighs the strict lower part twice):
        g_ell[l, k] = -(2 / ell_lk) sum_ij W_ij os dk/ds (z_ik - z_jk)^2,   g_os[l] = sum_ij W_ij k(s_ij),
        g_noise[l] = sum_i W_ii,   g_shape[l] = os sum_ij W_ij dk/dalpha.
    Returns a dict of these (float64 arrays), each with ``<name>_abs`` and ``<name>_prop`` (module docstring), for
    device distances bounded by ``ds_bound(..., dpad, expansion)``."""
    q, n, d = z.shape
    dpad = dpad or 4 * ((d + 3) // 4)
    out = {key: np.zeros((q, d)) for key in ("g_ell", "g_ell_abs", "g_ell_prop")}
    for key in ("g_os", "g_noise", "g_shape"):
        out[key], out[key + "_abs"], out[key + "_prop"] = np.zeros(q), np.zeros(q), np.zeros(q)
    for l in range(q):
        zl, Wl = z[l], W[l]
        a, o = _shape(alpha, l), _os(os_, l)
        nz = (zl * zl).sum(1)
        za = np.abs(zl)
        zt = torch.from_numpy(np.ascontiguousarray(zl))
        acc, prop_d = np.zeros(d), np.zeros(d)
        for i0, i1 in _blocks(n, n):
            s = sq_dist(zl[i0:i1], zl)
            ds = ds_bound(s, nz[i0:i1], nz, dpad, expansion)
            k, dk, dka, _ = profile(kid, s, a)
            Dk, Ddk, Ddka = _deltas(kid, s, ds, a)
            Wb = Wl[i0:i1]
            Wa = np.abs(Wb)
            A = torch.from_numpy(Wb * o * dk)
            P = torch.from_numpy(Wa * o * Ddk)
            for kk in range(d):                               # direct differences per dimension
                D2 = (zt[i0:i1, kk, None] - zt[None, :, kk]).square_()
                acc[kk] += float((A * D2).sum())
                prop_d[kk] += float((P * D2).sum())
            out["g_ell_abs"][l] += _abs_scale(Wa * o * (np.abs(dk) + Ddk), za[i0:i1], za)
            out["g_os"][l] += (Wb * k).sum()
            out["g_os_abs"][l] += (Wa * (k + Dk)).sum()
            out["g_os_prop"][l] += (Wa * Dk).sum()
            out["g_shape"][l] += o * (Wb * dka).sum()
            out["g_shape_abs"][l] += o * (Wa * (np.abs(dka) + Ddka)).sum()
            out["g_shape_prop"][l] += o * (Wa * Ddka).sum()
        f = 2.0 / np.asarray(ell[l], dtype=np.float64)
        out["g_ell"][l] = -f * acc
        out["g_ell_prop"][l] = f * prop_d
        out["g_ell_abs"][l] *= f
        diag = np.diagonal(Wl)
        out["g_noise"][l] = math.fsum(diag)
        out["g_noise_abs"][l] = np.abs(diag).sum()
    return out


def cross_gram_bwd(kid, zr, zc, G, ell, os_=None, alpha=None):
    """The adjoint of ``ops.cross_gram_bwd`` for K[l, i, j] = os_l k(|zr_li - zc_lj|^2) and the cotangent
    G [q, nr, nc]:
        g_ell[l, k] = -(2 / ell_lk) sum_ij G_ij os dk/ds (zr_ik - zc_jk)^2,   g_os[l] = sum_ij G_ij k,
        g_shape[l] = sum_ij G_ij os dk/dalpha,
        g_rows[i, k] = sum_l (2 / ell_lk) sum_j G_ij os dk/ds (zr_ik - zc_jk)   (w.r.t. the unscaled row points).
    Each with ``_abs`` and ``_prop`` as in ``sweep``; the device sums s by direct differences."""
    q, nr, d = zr.shape
    dpad = 4 * ((d + 3) // 4)
    out = {}
    for key, shape in (("g_ell", (q, d)), ("g_os", (q,)), ("g_shape", (q,)), ("g_rows", (nr, d))):
        for suf in ("", "_abs", "_prop"):
            out[key + suf] = np.zeros(shape)
    for l in range(q):
        a, o = _shape(alpha, l), _os(os_, l)
        s = sq_dist(zr[l], zc[l])
        ds = ds_bound(s, None, None, dpad, expansion=False)
        k, dk, dka, _ = profile(kid, s, a)
        Dk, Ddk, Ddka = _deltas(kid, s, ds, a)
        Gl = G[l]
        Ga = np.abs(Gl)
        A, P, E = Gl * o * dk, Ga * o * Ddk, Ga * o * (np.abs(dk) + Ddk)
        f = 2.0 / np.asarray(ell[l], dtype=np.float64)
        zra, zca = np.abs(zr[l]), np.abs(zc[l])
        for kk in range(d):
            D = zr[l][:, kk, None] - zc[l][None, :, kk]
            out["g_ell"][l, kk] = -f[kk] * (A * D * D).sum()
            out["g_ell_prop"][l, kk] = f[kk] * (P * D * D).sum()
            out["g_rows"][:, kk] += f[kk] * (A * D).sum(1)
            out["g_rows_prop"][:, kk] += f[kk] * (P * np.abs(D)).sum(1)
            out["g_rows_abs"][:, kk] += f[kk] * (zra[:, kk] * E.sum(1) + E @ zca[:, kk])
        out["g_ell_abs"][l] = f * _abs_scale(E, zra, zca)
        out["g_os"][l], out["g_os_abs"][l], out["g_os_prop"][l] = (Gl * k).sum(), (Ga * (k + Dk)).sum(), (Ga * Dk).sum()
        out["g_shape"][l] = o * (Gl * dka).sum()
        out["g_shape_abs"][l] = o * (Ga * (np.abs(dka) + Ddka)).sum()
        out["g_shape_prop"][l] = o * (Ga * Ddka).sum()
    return out
