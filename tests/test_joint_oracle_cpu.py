"""Joint predictive covariance of the oracle (CPU): the projected form sum_l C_l (x) h_l h_l^T + eps I against the dense
multitask model, its diagonal against the marginal prediction, its Gaussian log-density against scipy; argument checks
of the joint C-ABI entry points (no device needed)."""
import ctypes
import warnings

import pytest
import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import _cabi

from . import joint_reference as J
from .helpers import make_model, oracle_params, rel_err, synth


def _setup(variant, kernel, os_, ns=7):
    X, Y, Xs, Ys = synth(36, 2, 5, 2, seed=4, ns=ns)
    m = make_model(X, Y, 2, variant=variant, kernel=kernel, outputscales=os_)
    return X, Y, Xs, Ys, oracle_params(m)


@pytest.mark.parametrize("variant", ["PLMC", "PLMC_fast", "BDN_full"])
@pytest.mark.parametrize("kernel", ["rbf", "matern52"])
@pytest.mark.parametrize("os_", [False, True])
def test_joint_covariance_equals_dense_posterior_covariance(variant, kernel, os_):
    X, Y, Xs, _, p = _setup(variant, kernel, os_)
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        C, cov_f, cov_y = J.predict_joint(p, X, Y, Xs)
        dense = J.dense_posterior_covariance(p, X, Y, Xs)
        _, var_f, var_y = O.predict(p, X, Y, Xs)
    N = cov_f.shape[0]
    assert rel_err(cov_f - p.eps * torch.eye(N, dtype=cov_f.dtype), dense) < 1e-12
    assert rel_err(torch.diagonal(cov_f).reshape(var_f.shape), var_f) < 1e-12
    assert rel_err(torch.diagonal(cov_y).reshape(var_y.shape), var_y) < 1e-12
    assert C.shape == (p.q, Xs.shape[0], Xs.shape[0])


@pytest.mark.parametrize("full", [False, True])
def test_joint_log_density_equals_scipy(full):
    from scipy.stats import multivariate_normal

    X, Y, Xs, Ys, p = _setup("PLMC", "matern52", True, ns=9)
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mean, _, _ = O.predict(p, X, Y, Xs)
        _, cov_f, cov_y = J.predict_joint(p, X, Y, Xs)
    cov = cov_y if full else cov_f
    lp = O.mvn_log_prob(cov, (Ys - mean).reshape(-1))
    ref = multivariate_normal(mean=mean.reshape(-1).numpy(), cov=cov.numpy()).logpdf(Ys.reshape(-1).numpy())
    assert abs(lp.item() - ref) <= 1e-10 * abs(ref)


# ---- argument checks of the C ABI (host-side validation, before any device work) --------------------------------
def _lib():
    return _cabi.load()   # ctypes.CDLL of the in-tree library with the argument types of _cabi (no device)


FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below is rejected by its argument checks


def test_syrk_rejects_bad_arguments():
    lib = _lib()
    ok = (FAKE, 256, 256 * 256, FAKE, 256, 256 * 256, 256, 256, -1.0, 1.0, 1, None, None)
    for i, bad in [(0, None), (3, None), (6, 200), (7, 100), (7, 0), (1, 128), (4, 128), (10, 0)]:
        args = list(ok)
        args[i] = bad
        assert lib.plmc_syrk_batched(*args) == -1, (i, bad)


def test_task_covariance_rejects_bad_arguments():
    lib = _lib()
    ok = (FAKE, 16, 256, FAKE, FAKE, FAKE, 48, 10, 3, 2, 0, None)
    for i, bad in [(0, None), (3, None), (4, None), (5, None), (7, 0), (8, 0), (9, 0), (1, 5), (6, 20), (10, 2)]:
        args = list(ok)
        args[i] = bad
        assert lib.plmc_task_covariance(*args) == -1, (i, bad)
    tiled = list(ok)
    tiled[10] = 1
    tiled[6] = 30                       # the tiled form is of order npad(30) = 128
    assert lib.plmc_task_covariance(*tiled) == -1


def test_mix_samples_rejects_bad_arguments():
    lib = _lib()
    ok = (FAKE, FAKE, 128, 128 * 16, FAKE, FAKE, FAKE, FAKE, 10, 100, 3, 2, None)
    for i, bad in [(0, None), (1, None), (4, None), (5, None), (6, None), (7, None), (8, 0), (9, 0), (10, 0),
                   (11, 0), (2, 50)]:
        args = list(ok)
        args[i] = bad
        assert lib.plmc_mix_samples(*args) == -1, (i, bad)
