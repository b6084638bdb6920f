"""Joint eval-mode posterior on the GPU: covariance_matrix, rsample / sample and log_prob of the task-level
MultitaskMultivariateNormal, the latent covariances of compute_latent_distrib, against the CPU oracle."""
import warnings

import pytest
import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import distributed, ops
from projected_lmc_b200.engine import NanError

from . import joint_reference as J
from .helpers import cpu_copy, make_model, oracle_params, rel_err, synth

pytestmark = pytest.mark.gpu


def _case(variant="PLMC", kernel="rbf", os_=False, n=60, d=2, p=5, q=2, ns=37, seed=4, **extra):
    X, Y, Xs, Ys = synth(n, d, p, q, seed=seed, ns=ns)
    m = make_model(X, Y, q, variant=variant, kernel=kernel, outputscales=os_, **extra)
    po = oracle_params(cpu_copy(m))
    m = m.cuda()
    m.eval()
    return m, po, X, Y, Xs, Ys


def _oracle(po, X, Y, Xs):
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return J.predict_joint(po, X, Y, Xs)


def _check_parity(m, po, X, Y, Xs, tol=1e-7):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(Xs.cuda())
        full = m.full_likelihood()(pred)
    C, cov_f, cov_y = _oracle(po, X, Y, Xs)
    assert rel_err(pred.covariance_matrix, cov_f) < tol
    assert rel_err(full.covariance_matrix, cov_y) < tol
    return pred, full


@pytest.mark.parametrize("variant", ["PLMC", "PLMC_fast", "BDN_full", "oilmm"])
@pytest.mark.parametrize("kernel", ["rbf", "matern52", "matern32", "matern12"])
def test_covariance_matches_oracle(variant, kernel):
    _check_parity(*_case(variant, kernel)[:5])


@pytest.mark.parametrize("ns", [37, 300])
def test_covariance_with_outputscales(ns):
    _check_parity(*_case("PLMC", "matern52", os_=True, ns=ns)[:5])


def test_covariance_additive_kernel():
    _check_parity(*_case("PLMC", "matern52", n=90, d=4, ns=45, decomp=[[0, 1], [1, 2, 3]])[:5])


def test_latent_covariance_matches_oracle():
    m, po, X, Y, Xs, _ = _case("BDN_full", "matern32", os_=True)
    C, _, _ = _oracle(po, X, Y, Xs)
    lat = m.compute_latent_distrib(Xs.cuda())
    assert lat.covariance_matrix.shape == C.shape
    assert rel_err(lat.covariance_matrix, C) < 1e-7


@pytest.mark.parametrize("mode", ["rns", "digits"])
def test_covariance_on_the_int8_path(mode, capfd):
    """n = 2560, n* = 1024: V^T V (1024 x 1024 x 2560, lower, q = 2) runs on the INT8 tensor path."""
    m, po, X, Y, Xs, _ = _case("PLMC", "matern52", n=2560, d=4, p=6, ns=1024, seed=0)
    m._engine.gemm_mode = mode
    m._engine.rns_min_mnk = int(1e9)   # the default work floor sends a product of this size to digit planes
    ops.trace_enable(True)
    try:
        pred = m(Xs.cuda())
        T = pred.covariance_matrix
    finally:
        ops.trace_report()
        ops.trace_enable(False)
    report = capfd.readouterr().err.splitlines()
    syrk = [ln.split() for ln in report if ln.split()[1:6] == ["1024", "1024", "2560", "1", "2"]]
    assert syrk and all(r[0] == "int8" for r in syrk), report
    _, cov_f, _ = _oracle(po, X, Y, Xs)
    assert rel_err(T, cov_f) < 1e-7
    m._engine.gemm_mode = "fp64"
    m._pred_cache = None
    ref = m(Xs.cuda()).covariance_matrix
    assert rel_err(T, ref) < 1e-9


def test_fp32_grade_model():
    m, po, X, Y, Xs, _ = _case("PLMC_fast", "rbf")
    m = m.float()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(Xs.float().cuda())
    _, cov_f, _ = _oracle(po, X, Y, Xs)
    assert pred.covariance_matrix.dtype == torch.float32
    assert rel_err(pred.covariance_matrix, cov_f) < 1e-4


def test_consistency_with_the_marginal_prediction():
    m, po, X, Y, Xs, _ = _case("PLMC", "matern52", os_=True, ns=45)
    ops.stats_reset()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(Xs.cuda())
        full = m.full_likelihood()(pred)
    before = ops.stats_get()[0]
    for d in (pred, full):
        d.mean, d.variance, d.confidence_region()
    assert ops.stats_get()[0] == before          # marginals never launch the joint kernels
    T, Tf = pred.covariance_matrix, full.covariance_matrix
    assert torch.equal(T, T.T) and torch.equal(Tf, Tf.T)
    ns, p = pred.mean.shape
    assert rel_err(torch.diagonal(T).reshape(ns, p), pred._var) < 1e-12
    assert rel_err(torch.diagonal(Tf).reshape(ns, p), full._var) < 1e-12
    F = m.full_likelihood().task_noise_covar.detach()
    assert rel_err(Tf - T, torch.kron(torch.eye(ns, dtype=F.dtype, device=F.device), F)) < 1e-12


@pytest.mark.parametrize("full", [False, True])
def test_log_prob_matches_scipy(full):
    from scipy.stats import multivariate_normal

    m, po, X, Y, Xs, Ys = _case("BDN_full", "rbf", ns=30)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(Xs.cuda())
        if full:
            pred = m.full_likelihood()(pred)
    _, cov_f, cov_y = _oracle(po, X, Y, Xs)
    mvn = multivariate_normal(mean=pred.mean.cpu().reshape(-1).numpy(), cov=(cov_y if full else cov_f).numpy())
    g = torch.Generator().manual_seed(3)
    vals = Ys[None] + 0.3 * torch.randn((4,) + tuple(Ys.shape), generator=g, dtype=Ys.dtype)
    one = pred.log_prob(Ys.cuda())
    assert one.shape == ()
    assert abs(one.item() - mvn.logpdf(Ys.reshape(-1).numpy())) <= 1e-8 * abs(one.item())
    many = pred.log_prob(vals.cuda())
    ref = torch.as_tensor(mvn.logpdf(vals.reshape(4, -1).numpy()))
    assert many.shape == (4,)
    assert rel_err(many, ref) < 1e-8


def test_sample_latents_with_given_normals():
    m, po, X, Y, Xs, _ = _case("PLMC", "matern52", ns=40)
    C, _, _ = _oracle(po, X, Y, Xs)
    lat = m.compute_latent_distrib(Xs.cuda())
    g = torch.Generator().manual_seed(0)
    eps = torch.randn(2, 40, 6, generator=g, dtype=torch.float64)
    draws = lat._joint.sample_latents(eps.cuda())
    ref = torch.linalg.cholesky(C) @ eps + lat.mean.cpu()[:, :, None]
    assert rel_err(draws, ref) < 1e-7


def test_rsample_shapes_and_seed():
    m, po, X, Y, Xs, _ = _case("PLMC_fast", "rbf", ns=20)
    pred = m(Xs.cuda())
    assert pred.rsample().shape == (20, 5)
    assert pred.sample(torch.Size([2, 3])).shape == (2, 3, 20, 5)
    torch.cuda.manual_seed(11)
    a = pred.rsample(torch.Size([4]))
    torch.cuda.manual_seed(11)
    b = pred.rsample(torch.Size([4]))
    assert torch.equal(a, b)
    with pytest.raises(NotImplementedError):
        pred.rsample(torch.Size([2]), base_samples=torch.zeros(2, 20, 5, device="cuda"))


@pytest.mark.parametrize("full", [False, True])
def test_sample_statistics(full):
    m, po, X, Y, Xs, _ = _case("PLMC", "rbf", n=30, p=3, ns=16, seed=7)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(Xs.cuda())
        if full:
            pred = m.full_likelihood()(pred)
    S = 20000
    torch.cuda.manual_seed(5)
    s = pred.sample(torch.Size([S])).reshape(S, -1).double()
    cov = pred.covariance_matrix.double()
    mean = pred.mean.reshape(-1).double()
    se = (torch.diagonal(cov) / S).sqrt()
    assert ((s.mean(0) - mean).abs() <= 5 * se).all()
    emp = torch.cov(s.T)
    assert torch.linalg.norm(emp - cov) <= 0.05 * torch.linalg.norm(cov)


def test_singular_latent_covariance_gets_jitter():
    m, po, X, Y, Xs, _ = _case("PLMC", "rbf", ns=10)
    Xd = torch.cat([Xs, Xs, Xs[:1].expand(20, -1)]).cuda()
    pred = m(Xd)
    with pytest.warns(RuntimeWarning, match="jitter"):
        s = pred.rsample(torch.Size([8]))
    assert torch.isfinite(s).all()


def test_changed_parameter_is_an_error():
    m, po, X, Y, Xs, _ = _case()
    pred = m(Xs.cuda())
    lat = m.compute_latent_distrib(Xs.cuda())
    with torch.no_grad():
        m.likelihood.noise_covar.raw_noise.add_(0.1)
    with pytest.raises(RuntimeError, match="changed"):
        pred.covariance_matrix
    with pytest.raises(RuntimeError, match="changed"):
        lat.covariance_matrix


def test_rewritten_workspace_is_refactorised():
    m, po, X, Y, Xs, _ = _case()
    pred = m(Xs.cuda())
    m.compute_loo()
    _, cov_f, _ = _oracle(po, X, Y, Xs)
    assert rel_err(pred.covariance_matrix, cov_f) < 1e-7


def test_nan_test_point():
    m, po, X, Y, Xs, _ = _case(ns=12)
    Xn = Xs.clone()
    Xn[3, 0] = float("nan")
    pred = m(Xn.cuda())
    T = pred.covariance_matrix.view(12, 5, 12, 5)
    assert torch.isnan(T[3]).all() and torch.isnan(T[:, :, 3]).all()
    keep = [i for i in range(12) if i != 3]
    assert torch.isfinite(T[keep][:, :, keep]).all()
    with pytest.raises(NanError):
        pred.rsample()
    with pytest.raises(NanError):
        pred.log_prob(torch.zeros(12, 5, dtype=torch.float64, device="cuda"))


def test_unsupported_models():
    m, po, X, Y, Xs, _ = _case(n_inducing_points=16)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(Xs.cuda())
    with pytest.raises(NotImplementedError, match="SGPR"):
        pred.covariance_matrix
    m, po, X, Y, Xs, _ = _case()
    distributed.shard_latents(m, rank=0, world=2)
    pred = m(Xs.cuda())
    with pytest.raises(NotImplementedError, match="sharded"):
        pred.rsample()
