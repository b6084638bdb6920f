"""Gradients of eval-mode predictions w.r.t. the test inputs on the GPU: x.grad of model(x).mean / .variance (and of
compute_latent_distrib and full_likelihood()(pred)) against torch autograd through the CPU oracle, the INT8 routes
of the variance backward, bit-identity of the forward, determinism, stale states, non-finite rows, and the fused
cross_grad kernel against the composed SGPR-adjoint path."""
import warnings

import pytest
import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import ops

from . import input_grad_reference as R
from .helpers import cpu_copy, make_model, rel_err, synth
from .rq_reference import rq_kernels

pytestmark = pytest.mark.gpu

TOL = 1e-7


def _case(variant="PLMC", kernel="rbf", os_=False, n=80, d=3, p=5, q=2, ns=37, seed=4, **extra):
    X, Y, Xs, _ = synth(n, d, p, q, seed=seed, ns=ns)
    if kernel == "rq":
        m = R.rq_model(X, Y, q, outputscales=os_, seed=seed, **extra)
    else:
        m = make_model(X, Y, q, variant=variant, kernel=kernel, outputscales=os_, **extra)
    po, raw = R.oracle_params_and_alphas(cpu_copy(m))
    m = m.cuda()
    m.eval()
    return m, po, raw, X, Y, Xs


def _weights(ns, p, seed=7):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(ns, p, generator=g, dtype=torch.float64),
            torch.randn(ns, p, generator=g, dtype=torch.float64))


def _model_grad(m, Xs, Wm, Wv, full=False, dtype=torch.float64):
    x = Xs.to(dtype).cuda().requires_grad_(True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(x)
        if full:
            pred = m.full_likelihood()(pred)
    f = 0.0
    if Wm is not None:
        f = f + (pred.mean * Wm.to(dtype).cuda()).sum()
    if Wv is not None:
        f = f + (pred.variance * Wv.to(dtype).cuda()).sum()
    f.backward()
    return x.grad


def _oracle_grad(po, raw, X, Y, Xs, Wm, Wv, which=1):
    with (rq_kernels(raw) if raw is not None else warnings.catch_warnings()):
        warnings.simplefilter("ignore")
        return R.autograd_input_grad(po, X, Y, Xs, Wm, Wv, which)


@pytest.mark.parametrize("variant", ["PLMC", "PLMC_fast", "BDN_full", "oilmm"])
@pytest.mark.parametrize("kernel", ["rbf", "matern52", "matern32", "matern12"])
def test_grad_matches_oracle(variant, kernel):
    m, po, raw, X, Y, Xs = _case(variant, kernel)
    Wm, Wv = _weights(*Xs.shape[:1], Y.shape[1])
    assert rel_err(_model_grad(m, Xs, Wm, Wv), _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < TOL


@pytest.mark.parametrize("kernel", ["matern52", "rq"])
@pytest.mark.parametrize("which", ["mean", "var", "both"])
def test_grad_with_outputscales_and_decomp(kernel, which):
    m, po, raw, X, Y, Xs = _case("PLMC", kernel, os_=True, n=90, d=4, ns=45, decomp=[[0, 1], [1, 2, 3]])
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    Wm, Wv = (Wm if which != "var" else None), (Wv if which != "mean" else None)
    assert rel_err(_model_grad(m, Xs, Wm, Wv), _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < TOL


@pytest.mark.parametrize("os_", [False, True])
def test_rq_grad(os_):
    m, po, raw, X, Y, Xs = _case("PLMC", "rq", os_=os_)
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    assert rel_err(_model_grad(m, Xs, Wm, Wv), _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < TOL


def test_compute_latent_distrib_grad():
    m, po, raw, X, Y, Xs = _case("BDN_full", "matern32", os_=True)
    g = torch.Generator().manual_seed(2)
    Wm = torch.randn(2, Xs.shape[0], generator=g, dtype=torch.float64)
    Wv = torch.randn(2, Xs.shape[0], generator=g, dtype=torch.float64)
    x = Xs.cuda().requires_grad_(True)
    lat = m.compute_latent_distrib(x)
    ((lat.mean * Wm.cuda()).sum() + (lat.stddev.pow(2) * Wv.cuda()).sum()).backward()
    xs = Xs.clone().requires_grad_(True)
    lm, lv = R.latent_predict(po, X, Y, xs)
    (ref,) = torch.autograd.grad((lm * Wm).sum() + (lv * Wv).sum(), xs)
    assert rel_err(x.grad, ref) < TOL


def test_full_likelihood_grad():
    m, po, raw, X, Y, Xs = _case("PLMC", "rbf", os_=True)
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    assert rel_err(_model_grad(m, Xs, Wm, Wv, full=True), _oracle_grad(po, raw, X, Y, Xs, Wm, Wv, which=2)) < TOL


@pytest.mark.parametrize("kernel", ["rbf", "matern52"])
def test_sgpr_grad(kernel):
    m, po, raw, X, Y, Xs = _case("PLMC", kernel, os_=True, n=300, d=3, ns=70, n_inducing_points=40, seed=8)
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    assert rel_err(_model_grad(m, Xs, Wm, Wv), _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < TOL


@pytest.mark.parametrize("mode", ["fp64", "rns", "digits"])
@pytest.mark.parametrize("inverse", [False, True])
def test_int8_paths_over_several_tiles(mode, inverse, capfd):
    """n = 2560, n* = 1000 in tiles of 384: the two triangular products of each tile take the INT8 tensor path."""
    m, po, raw, X, Y, Xs = _case("PLMC", "matern52", n=2560, d=4, p=6, ns=1000, seed=0)
    eng = m._engine
    eng.gemm_mode = mode
    eng.rns_min_mnk = int(1e8)
    eng.predict_inverse = inverse
    eng.tile_points = lambda *a, **k: 384
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    x = Xs.cuda().requires_grad_(True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(x)
    f = (pred.mean * Wm.cuda()).sum() + (pred.variance * Wv.cuda()).sum()
    capfd.readouterr()
    ops.trace_enable(True)
    try:
        f.backward()
    finally:
        ops.trace_report()
        ops.trace_enable(False)
    report = [ln.split() for ln in capfd.readouterr().err.splitlines() if ln.strip()]
    assert bool(m._pred_cache.get("inverted")) == inverse
    if mode != "fp64":     # "tri": a residue-mode triangular product as one INT8 launch set
        assert any(r[0] in ("int8", "tri") for r in report), report
    assert rel_err(x.grad, _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < TOL


def test_fp32_model():
    m, po, raw, X, Y, Xs = _case("PLMC_fast", "rbf")
    m = m.float()
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    g = _model_grad(m, Xs, Wm, Wv, dtype=torch.float32)
    assert g.dtype == torch.float32
    assert rel_err(g, _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < 1e-4


def test_one_dimensional_inputs():
    m, po, raw, X, Y, Xs = _case("PLMC", "matern52", d=1)
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    x = Xs[:, 0].cuda().requires_grad_(True)
    pred = m(x)
    ((pred.mean * Wm.cuda()).sum() + (pred.stddev * Wv.cuda()).sum()).backward()
    assert x.grad.shape == x.shape
    xs = Xs.clone().requires_grad_(True)
    mean, var_f, _ = O.predict(po, X, Y, xs)
    (ref,) = torch.autograd.grad((mean * Wm).sum() + (var_f.sqrt() * Wv).sum(), xs)
    assert rel_err(x.grad, ref[:, 0]) < TOL


@pytest.mark.parametrize("kernel", ["rbf", "matern52", "matern32", "rq"])
def test_test_point_on_a_training_point(kernel):
    m, po, raw, X, Y, Xs = _case("PLMC", kernel)
    Xs = Xs.clone()
    Xs[3] = X[5]
    Xs[10] = X[0]
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    assert rel_err(_model_grad(m, Xs, Wm, Wv), _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < TOL


def test_forward_is_bit_identical_and_backward_deterministic():
    m, po, raw, X, Y, Xs = _case("PLMC", "matern52", os_=True, n=700, decomp=[[0, 1], [1, 2]])
    m._engine.predict_inverse = False     # "auto" would invert the state between the calls below
    with torch.no_grad():
        ref = m(Xs.cuda())
        lat_ref = m.compute_latent_distrib(Xs.cuda())
    x = Xs.cuda().requires_grad_(True)
    pred = m(x)
    lat = m.compute_latent_distrib(x)
    assert pred.mean.requires_grad and lat.mean.requires_grad
    assert torch.equal(pred.mean, ref.mean) and torch.equal(pred.variance, ref.variance)
    assert torch.equal(lat.mean, lat_ref.mean) and torch.equal(lat.variance, lat_ref.variance)
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    g1, g2 = (_model_grad(m, Xs, Wm, Wv) for _ in range(2))
    assert torch.equal(g1, g2)


def test_mean_only_backward_launches_no_triangular_op():
    m, po, raw, X, Y, Xs = _case("PLMC", "rbf", n=300, ns=200, decomp=[[0, 1], [1, 2]])
    m._engine.tile_points = lambda *a, **k: 128
    x = Xs.cuda().requires_grad_(True)
    pred = m(x)
    f = pred.mean.sum()
    ops.stats_reset()
    f.backward()
    # mix_tasks_bwd, then per tile (2) and component (2): scale_inputs + cross_grad (kernel + reduction)
    assert ops.stats_get()[0] == 1 + 2 * 2 * 3
    Wm = torch.ones(Xs.shape[0], Y.shape[1], dtype=torch.float64)
    assert rel_err(x.grad, _oracle_grad(po, raw, X, Y, Xs, Wm, None)) < TOL


def test_stale_states():
    m, po, raw, X, Y, Xs = _case("PLMC", "matern52")
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    x = Xs.cuda().requires_grad_(True)
    pred = m(x)
    f = (pred.mean * Wm.cuda()).sum() + (pred.variance * Wv.cuda()).sum()
    m.compute_loo()                       # rewrites the engine workspace: the backward re-factorises
    f.backward()
    assert rel_err(x.grad, _oracle_grad(po, raw, X, Y, Xs, Wm, Wv)) < TOL
    pred = m(Xs.cuda().requires_grad_(True))
    f = pred.variance.sum()
    with torch.no_grad():
        m.likelihood.noise_covar.raw_noise.add_(0.1)
    with pytest.raises(RuntimeError, match="changed after this prediction"):
        f.backward()


def test_non_finite_rows():
    m, po, raw, X, Y, Xs = _case("PLMC", "rbf")
    Wm, Wv = _weights(Xs.shape[0], Y.shape[1])
    ref = _model_grad(m, Xs, Wm, Wv)
    Xb = Xs.clone()
    Xb[4, 1] = float("nan")
    Xb[9, 0] = float("inf")
    x = Xb.cuda().requires_grad_(True)
    pred = m(x)
    f = (pred.mean * Wm.cuda()).nan_to_num().sum() + (pred.variance * Wv.cuda()).nan_to_num().sum()
    f.backward()
    bad = torch.zeros(Xs.shape[0], dtype=torch.bool)
    bad[4] = bad[9] = True
    assert torch.isnan(x.grad[bad.cuda()]).all()
    assert rel_err(x.grad[~bad.cuda()], ref[~bad.cuda()]) < 1e-12


@pytest.mark.parametrize("kid", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("d", [3, 21, 30])
def test_cross_grad_against_the_composed_adjoint(kid, d):
    """plmc_cross_grad against w materialised as the cotangent of the cross block, with the test points as its rows,
    through plmc_cross_gram_bwd2; garbage in the padding columns of beta changes nothing."""
    g = torch.Generator().manual_seed(kid + d)
    q, n, ns = 3, 700, 333
    dev = "cuda"
    X = (torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
    Xs = (torch.rand(ns, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
    ell = (0.5 + torch.rand(q, d, generator=g, dtype=torch.float64)).to(dev)
    os_ = (0.5 + torch.rand(q, generator=g, dtype=torch.float64)).to(dev)
    shape = (0.5 + torch.rand(q, generator=g, dtype=torch.float64)).to(dev) if kid == 4 else None
    alpha = torch.randn(q, n, generator=g, dtype=torch.float64).to(dev)
    gm = torch.randn(q, ns, generator=g, dtype=torch.float64).to(dev)
    gv = torch.randn(q, ns, generator=g, dtype=torch.float64).to(dev)
    xm = ops.col_mean(X)
    np_, mt = ops.npad(n), ops.npad(ns)
    Z, zn = ops.scale_inputs(X, xm, ell, np_)
    Zt, znt = ops.scale_inputs(Xs, xm, ell, mt)
    beta = torch.full((q, np_, mt), float("nan"), dtype=torch.float64, device=dev)
    beta[:, :n, :ns] = torch.randn(q, n, ns, generator=g, dtype=torch.float64).to(dev)
    beta[:, n:, :ns] = 0.0
    got = ops.cross_grad(Z, zn, Zt, znt, kid, os_, ell, alpha, n, ns, gm, gv, beta, shape=shape)
    got_m = ops.cross_grad(Z, zn, Zt, znt, kid, os_, ell, alpha, n, ns, gm, None, None, shape=shape)
    for gvv, out in ((gv, got), (None, got_m)):
        w = gm[:, None, :] * alpha[:, :, None]
        if gvv is not None:
            w = w - 2 * gvv[:, None, :] * beta[:, :n, :ns]
        G = w.transpose(1, 2).contiguous()                  # [q, ns, n]: test points as rows
        ref = ops.cross_gram_bwd(Zt, Z, G, kid, os_, ell, ns, n, shape=shape)[2]
        assert rel_err(out, ref) < 1e-12
    assert torch.equal(got, ops.cross_grad(Z, zn, Zt, znt, kid, os_, ell, alpha, n, ns, gm, gv, beta, shape=shape))


def test_mix_tasks_bwd_against_torch():
    g = torch.Generator().manual_seed(0)
    q, p, ns = 3, 7, 301
    H = torch.randn(q, p, generator=g, dtype=torch.float64).cuda()
    gm = torch.randn(ns, p, generator=g, dtype=torch.float64).cuda()
    gv = torch.randn(ns, p, generator=g, dtype=torch.float64).cuda()
    a, b = ops.mix_tasks_bwd(H, gm, gv)
    assert rel_err(a, (gm @ H.T).T) < 1e-14 and rel_err(b, (gv @ H.pow(2).T).T) < 1e-14
    a2, b2 = ops.mix_tasks_bwd(H, None, gv)
    assert a2 is None and torch.equal(b2, b)
