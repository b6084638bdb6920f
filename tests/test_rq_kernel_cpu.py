"""Rational quadratic kernel (gpytorch RQKernel) without a GPU: the hand-written log1p and the RQ profile of
csrc/kernel_math.cuh on the host, the CPU reference of tests/rq_reference.py against scikit-learn and against the
trace formula of its alpha gradient, the model surface, and the argument checks of the shaped C ABI entry points."""
import ctypes
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import ProjectedGPModel, _cabi, gp, ops

from .helpers import synth
from .rq_reference import rq_kernel, rq_kernels

P = ctypes.c_void_p


def _p(a):
    return None if a is None else a.ctypes.data_as(P)


def log1p_host(x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    assert _cabi.load().plmc_log1p_host(_p(x), x.size, _p(out)) == 0
    return out


def profile2(kid, s, alpha=None):
    s = np.ascontiguousarray(s, dtype=np.float64)
    k, dk, da = np.empty_like(s), np.empty_like(s), np.empty_like(s)
    a = None if alpha is None else np.ascontiguousarray(np.broadcast_to(alpha, s.shape), dtype=np.float64)
    rc = _cabi.load().plmc_kernel_profile2_host(kid, _p(s), _p(a), s.size, _p(k), _p(dk), _p(da))
    assert rc == 0
    return k, dk, da


def ulps(got, ref):
    """|got - ref| in units of the last place of ref (ref in extended precision)."""
    sp = np.spacing(np.abs(ref.astype(np.float64)))
    sp = np.where(sp > 0, sp, np.finfo(np.float64).smallest_subnormal)
    return np.abs(got.astype(np.longdouble) - ref) / sp


def test_log1p_is_within_1p2_ulp_of_the_correctly_rounded_value():
    rng = np.random.default_rng(0)
    x = np.concatenate([10.0 ** rng.uniform(-300, 15, 100000), 10.0 ** rng.uniform(-12, 6, 100000),
                        rng.uniform(0, 3, 100000), [0.0, 5e-324, 1e-300, 0.5, 1.0, 2.0, 1e15, 1e300]])
    got = log1p_host(x)
    ref = np.log1p(x.astype(np.longdouble))            # 64-bit mantissa: exact to ~1/2000 of a double ulp
    assert got[np.where(x == 0)[0][0]] == 0.0
    assert ulps(got, ref).max() < 1.2


def rq_reference(s, a):
    """k, dk/ds, dk/dalpha of (1 + s / (2 alpha))^-alpha in extended precision."""
    s, a = s.astype(np.longdouble), a.astype(np.longdouble)
    x = s / (2 * a)
    b = 1 + x
    L = np.log1p(x)
    k = np.exp(-a * L)
    return k, -0.5 * k / b, k * (x / b - L)


def test_rq_profile_against_the_closed_form():
    rng = np.random.default_rng(1)
    s = np.concatenate([[0.0], 10.0 ** rng.uniform(-12, 3, 40000), rng.uniform(0, 1e3, 20000)])
    a = 10.0 ** rng.uniform(-2, 8, s.size)
    k, dk, da = profile2(ops.KERNEL_RQ, s, a)
    kr, dkr, dar = rq_reference(s, a)
    # k = exp(-alpha L) amplifies a relative rounding of alpha L, of x = s / (2 alpha) and of L by alpha L (<= s/2).
    # A double evaluation of the formula with numpy's exp / log1p reaches 2.3 (alpha L + 1) ulp on these points; the
    # kernel's hand-written log1p / exp / reciprocal stay within 3 (alpha L + 1)
    cond = (a * np.log1p(s / (2 * a)) + 1.0).astype(np.longdouble)
    assert (ulps(k, kr) / cond).max() < 3.0
    assert (ulps(dk, dkr) / cond).max() < 3.0
    # dk/dalpha = k (x / b - L): 1e-15 absolute, relative where |dk/dalpha| exceeds 1 (small alpha)
    dar = dar.astype(np.float64)
    assert (np.abs(da - dar) / np.maximum(1.0, np.abs(dar))).max() < 1e-15
    # at s = 0: k = 1, both derivatives of the diagonal as gpytorch's autograd gives them (dk/ds = -1/2, dk/dalpha = 0)
    assert k[0] == 1.0 and dk[0] == -0.5 and da[0] == 0.0


def test_rq_approaches_rbf_at_large_alpha():
    s = np.linspace(0.0, 60.0, 2001)
    k, dk, da = profile2(ops.KERNEL_RQ, s, 1e8)
    kr, dkr, _ = profile2(0, s)
    assert np.abs(k - kr).max() < 1e-7
    assert np.abs(dk - dkr).max() < 1e-7
    assert np.abs(da).max() < 1e-7


def test_profile2_for_kernels_0_to_3_matches_the_old_entry_point_bit_for_bit():
    lib = _cabi.load()
    s = np.concatenate([[0.0], 10.0 ** np.random.default_rng(2).uniform(-8, 3, 5000)])
    for kid in range(4):
        k0, dk0 = np.empty_like(s), np.empty_like(s)
        assert lib.plmc_kernel_profile_host(kid, _p(s), s.size, _p(k0), _p(dk0)) == 0
        k, dk, da = profile2(kid, s)
        assert np.array_equal(k, k0) and np.array_equal(dk, dk0) and not da.any()


def test_shaped_abi_argument_checks():
    lib = _cabi.load()
    BAD = -1
    s = np.ones(4)
    out = [np.empty(4) for _ in range(3)]
    alpha = np.ones(4)
    # RQ without a shape, a shape for kernels 0-3
    assert lib.plmc_kernel_profile2_host(ops.KERNEL_RQ, _p(s), None, 4, *map(_p, out)) == BAD
    assert lib.plmc_kernel_profile2_host(1, _p(s), _p(alpha), 4, *map(_p, out)) == BAD
    assert lib.plmc_kernel_profile2_host(5, _p(s), _p(alpha), 4, *map(_p, out)) == BAD
    # the device entry points refuse the same combinations before touching any pointer (host addresses here)
    Z, zn, K = np.zeros(128 * 4), np.zeros(128), np.zeros(128 * 128)
    os_, da = np.ones(1), np.zeros(1)
    for kid, shape in ((ops.KERNEL_RQ, None), (0, alpha), (3, alpha)):
        assert lib.plmc_gram2(_p(Z), _p(zn), kid, _p(os_), _p(shape), _p(da), _p(K), 128, 0, 100, 128, 4, 1, 0,
                              None) == BAD
        assert lib.plmc_cross_gram2(_p(Z), _p(zn), _p(Z), _p(zn), kid, _p(os_), _p(shape), _p(K), 128, 0, 100, 128,
                                    128, 128, 4, 1, 0, None) == BAD
        g = [np.zeros(4) for _ in range(4)]
        ws = np.zeros(4096)
        assert lib.plmc_grad_sweep2(_p(K), 128, 0, _p(zn), 128, _p(Z), _p(zn), _p(os_), kid, _p(os_), _p(shape),
                                    _p(g[0]), _p(g[1]), _p(g[2]), _p(g[3]), _p(ws), 100, 128, 4, 4, 1, None) == BAD
        assert lib.plmc_cross_gram_bwd2(_p(Z), 128, _p(Z), 128, _p(K), 128, 0, kid, _p(os_), _p(shape), _p(os_),
                                        _p(g[0]), _p(g[1]), _p(g[3]), _p(g[2]), _p(ws), 100, 100, 4, 4, 1, None) == BAD
    # g_shape without a shape
    g = [np.zeros(4) for _ in range(4)]
    ws = np.zeros(4096)
    assert lib.plmc_grad_sweep2(_p(K), 128, 0, _p(zn), 128, _p(Z), _p(zn), _p(os_), 0, _p(os_), None, _p(g[0]),
                                _p(g[1]), _p(g[2]), _p(g[3]), _p(ws), 100, 128, 4, 4, 1, None) == BAD
    assert lib.plmc_cross_gram_bwd2(_p(Z), 128, _p(Z), 128, _p(K), 128, 0, 0, _p(os_), None, _p(os_), _p(g[0]),
                                    _p(g[1]), _p(g[3]), _p(g[2]), _p(ws), 100, 100, 4, 4, 1, None) == BAD
    # workspaces: one more accumulator per latent and CTA for RQ
    assert lib.plmc_grad_ws2(1024, 5, 3, 0) == lib.plmc_grad_ws(1024, 5, 3)
    assert lib.plmc_grad_ws2(1024, 5, 3, ops.KERNEL_RQ) == lib.plmc_grad_ws(1024, 5, 3) // 10 * 11
    assert lib.plmc_cross_gram_bwd_ws2(300, 5000, 5, 2, 1) == lib.plmc_cross_gram_bwd_ws(300, 5000, 5, 2)
    assert lib.plmc_cross_gram_bwd_ws2(300, 5000, 5, 2, ops.KERNEL_RQ) > lib.plmc_cross_gram_bwd_ws(300, 5000, 5, 2)


@pytest.mark.parametrize("alpha", [0.05, 0.7, 3.0, 40.0])
def test_rq_reference_matches_scikit_learn(alpha):
    from sklearn.gaussian_process.kernels import RationalQuadratic

    g = torch.Generator().manual_seed(3)
    X1 = torch.rand(40, 3, generator=g) * 4 - 2
    X2 = torch.rand(25, 3, generator=g) * 4 - 2
    ell = 0.8
    K = rq_kernel(X1, X2, torch.full((1, 1, 3), ell), zero_diag=False, alpha=torch.tensor([[alpha]]))
    ref = RationalQuadratic(length_scale=ell, alpha=alpha)(X1.numpy(), X2.numpy())
    assert np.abs(K[0].numpy() - ref).max() < 1e-13


def test_reference_alpha_gradient_against_the_trace_formula():
    g = torch.Generator().manual_seed(4)
    n, d, q = 30, 2, 2
    X = torch.rand(n, d, generator=g) * 2 - 1
    TY = torch.randn(q, n, generator=g)
    raw_alpha = torch.tensor([[-0.4], [1.3]], requires_grad=True)
    p = O.OracleParams(raw_lengthscale=torch.tensor([[[0.2, -0.3]], [[0.5, 0.1]]]), raw_noise=torch.full((q, 1), -2.0),
                       noise_lower=1e-4, kernel="rq", raw_outputscale=torch.tensor([0.3, -0.2]))
    with rq_kernels([raw_alpha]):
        lp = O.latent_log_probs(p, X, TY)
    grad, = torch.autograd.grad(lp.sum(), raw_alpha)
    with torch.no_grad():
        a = O.softplus(raw_alpha).reshape(q, 1, 1)
        s = O.sq_dist(X / O.lengthscale(p), X / O.lengthscale(p), zero_diag=False)
        k = (1 + s / (2 * a)) ** (-a)
        dk_da = k * (s / (2 * a + s) - torch.log1p(s / (2 * a))) * O.outputscale(p)[:, None, None]
        K = O.outputscale(p)[:, None, None] * k + torch.diag_embed(O.noise(p)[:, None].expand(-1, n))
        Kinv = torch.linalg.inv(K)
        al = (Kinv @ TY.unsqueeze(-1))
        W = al @ al.transpose(1, 2) - Kinv
        g_alpha = 0.5 * (W * dk_da).sum((1, 2))
        ref = g_alpha * torch.sigmoid(raw_alpha.squeeze(-1))      # softplus'
    assert torch.allclose(grad.squeeze(-1), ref, rtol=1e-10, atol=1e-12)


def _rq_model(decomp=None, outputscales=False, **kw):
    X, Y, _, _ = synth(30, 3, 4, 2)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ProjectedGPModel(X, Y, 4, 2, mean_type=gp.means.ZeroMean, kernel_type=gp.kernels.RQKernel, decomp=decomp,
                                outputscales=outputscales, **kw)


def test_rq_model_surface():
    m = _rq_model()
    base = m._base_kernel()
    assert isinstance(base, gp.kernels.RQKernel) and base.kernel_id == 4
    assert base.raw_alpha.shape == (2, 1)
    assert torch.allclose(base.alpha, torch.full((2, 1), math.log(2.0)))
    base.alpha = torch.tensor([[0.5], [3.0]])
    assert torch.allclose(base.alpha, torch.tensor([[0.5], [3.0]]))
    assert "covar_module.raw_alpha" in m.state_dict()
    assert "covar_module.base_kernel.raw_alpha" in _rq_model(outputscales=True).state_dict()
    sd = _rq_model(decomp=[[0, 1], [1, 2]]).state_dict()
    assert "covar_module.kernels.0.base_kernel.raw_alpha" in sd and "covar_module.kernels.1.base_kernel.raw_alpha" in sd
    # lscales() / outputscale() are those of any other ARD kernel
    assert m.lscales().shape == (2, 3)
    mo = _rq_model(outputscales=True)
    assert torch.allclose(mo.outputscale(), torch.full((2, 1), math.log(2.0)))
    # a constraint of the caller's choice
    mc = _rq_model(ker_kwargs={"alpha_constraint": gp.constraints.GreaterThan(0.5)})
    assert torch.allclose(mc._base_kernel().alpha, torch.full((2, 1), 0.5 + math.log(2.0)))
    # components carry alpha beside the (kid, dims, ell, os) tuple; the other kernels keep plain tuples' behaviour
    comp, = m._kernel_components()
    kid, dims, ell, os_ = comp
    assert kid == 4 and os_ is None and torch.equal(ops.shape_of(comp), base.alpha.squeeze(-1))
    spec, tensors = m._local_components()
    assert spec == ((4, (0, 1, 2), False, True),) and len(tensors) == 2


def test_kernel_type_resolved_from_a_foreign_class_name():
    class RQKernel:      # stands for gpytorch.kernels.RQKernel: resolution is by class name
        pass

    X, Y, _, _ = synth(20, 2, 3, 2)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = ProjectedGPModel(X, Y, 3, 2, mean_type=gp.means.ZeroMean, kernel_type=RQKernel)
    assert isinstance(m._base_kernel(), gp.kernels.RQKernel)
