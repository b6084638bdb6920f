"""Gradients of eval-mode predictions w.r.t. the test inputs without a GPU: the closed form of
tests/input_grad_reference.py against torch autograd through the oracle and against central finite differences,
for every kernel, outputscales, an additive kernel with overlapping active dims, mean-only / variance-only /
combined cotangents and the mixing adjoint; argument checks of the C entry points; DMMA in the SASS of the kernel."""
import ctypes
import shutil
import subprocess
import warnings

import pytest
import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import _cabi

from . import input_grad_reference as R
from .helpers import make_model, rel_err, synth
from .rq_reference import rq_kernels

KERNELS = ["rbf", "matern52", "matern32", "matern12", "rq"]


def _setup(kernel, os_=False, decomp=None, n=40, d=3, p=4, q=2, ns=9):
    X, Y, Xs, _ = synth(n, d, p, q, seed=5, ns=ns)
    extra = {} if decomp is None else dict(decomp=decomp)
    if kernel == "rq":
        m = R.rq_model(X, Y, q, outputscales=os_, **extra)
    else:
        m = make_model(X, Y, q, kernel=kernel, outputscales=os_, **extra)
    po, raw = R.oracle_params_and_alphas(m)
    return po, raw, X, Y, Xs


def _ctx(raw):
    return rq_kernels(raw) if raw is not None else warnings.catch_warnings()


def _cotangents(ns, p, which, seed=3):
    g = torch.Generator().manual_seed(seed)
    gm = torch.randn(ns, p, generator=g, dtype=torch.float64)
    gv = torch.randn(ns, p, generator=g, dtype=torch.float64)
    return (gm if which in ("mean", "both") else None), (gv if which in ("var", "both") else None)


def _alphas(raw):
    return None if raw is None else [O.softplus(r).detach().reshape(-1) for r in raw]


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("os_", [False, True])
def test_closed_form_equals_oracle_autograd(kernel, os_):
    po, raw, X, Y, Xs = _setup(kernel, os_)
    gm, gv = _cotangents(Xs.shape[0], Y.shape[1], "both")
    with _ctx(raw):
        ref = R.autograd_input_grad(po, X, Y, Xs, gm, gv)
        got = R.input_grad(po, X, Y, Xs, gm, gv, _alphas(raw))
    assert rel_err(got, ref) < 1e-10


@pytest.mark.parametrize("which", ["mean", "var", "both"])
@pytest.mark.parametrize("kernel", ["matern52", "rq"])
def test_cotangent_kinds_and_additive_kernel(which, kernel):
    po, raw, X, Y, Xs = _setup(kernel, True, decomp=[[0, 1], [1, 2]])
    gm, gv = _cotangents(Xs.shape[0], Y.shape[1], which)
    with _ctx(raw):
        ref = R.autograd_input_grad(po, X, Y, Xs, gm, gv)
        got = R.input_grad(po, X, Y, Xs, gm, gv, _alphas(raw))
    assert rel_err(got, ref) < 1e-10


@pytest.mark.parametrize("kernel", KERNELS)
def test_closed_form_equals_central_differences(kernel):
    po, raw, X, Y, Xs = _setup(kernel, True, decomp=[[0, 1], [1, 2]], ns=5)
    gm, gv = _cotangents(Xs.shape[0], Y.shape[1], "both")
    h = 1e-5
    with _ctx(raw), torch.no_grad():
        got = R.input_grad(po, X, Y, Xs, gm, gv, _alphas(raw))

        def f(xs):
            mean, var_f, _ = O.predict(po, X, Y, xs)
            return ((mean * gm).sum() + (var_f * gv).sum()).item()

        fd = torch.zeros_like(Xs)
        for j in range(Xs.shape[0]):
            for k in range(Xs.shape[1]):
                e = torch.zeros_like(Xs)
                e[j, k] = h
                fd[j, k] = (f(Xs + e) - f(Xs - e)) / (2 * h)
    assert rel_err(got, fd) < 1e-6


def test_full_likelihood_variance_has_the_same_gradient():
    po, raw, X, Y, Xs = _setup("rbf", True)
    gm, gv = _cotangents(Xs.shape[0], Y.shape[1], "both")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = R.autograd_input_grad(po, X, Y, Xs, gm, gv, which=2)
    assert rel_err(R.input_grad(po, X, Y, Xs, gm, gv), ref) < 1e-10


def test_mixing_adjoint_equals_autograd():
    g = torch.Generator().manual_seed(1)
    q, p, ns = 3, 5, 11
    H = torch.randn(q, p, generator=g, dtype=torch.float64)
    lm = torch.randn(q, ns, generator=g, dtype=torch.float64, requires_grad=True)
    lv = torch.randn(q, ns, generator=g, dtype=torch.float64, requires_grad=True)
    gm, gv = _cotangents(ns, p, "both")
    f = ((lm.T @ H) * gm).sum() + ((lv.T @ H.pow(2)) * gv).sum()
    rm, rv = torch.autograd.grad(f, (lm, lv))
    am, av = R.mixing_adjoint(H, gm, gv)
    assert rel_err(am, rm) < 1e-14 and rel_err(av, rv) < 1e-14
    assert R.mixing_adjoint(H, None, gv)[0] is None and R.mixing_adjoint(H, gm, None)[1] is None


# ---- argument checks of the C ABI (host-side validation, before any device work) --------------------------------
FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below is rejected by its argument checks


def test_cross_grad_rejects_bad_arguments():
    lib = _cabi.load()
    #     Ztr   zntr  npad Zte   znte  rpt  kid os    shape ell   alpha lda  gm    gv    ldg  beta  ldb  strideb
    ok = [FAKE, FAKE, 256, FAKE, FAKE, 128, 1, None, None, FAKE, FAKE, 250, FAKE, FAKE, 100, FAKE, 128, 256 * 128,
          FAKE, 3, FAKE, 250, 100, 3, 4, 2, None]
    #     g_x   ldx partial n  ns   d  dpad q stream
    cases = [(0, None), (1, None), (3, None), (4, None), (9, None), (10, None), (18, None), (20, None), (2, 200),
             (2, 128), (5, 64), (6, 5), (6, -1), (6, 4), (8, FAKE), (11, 100), (13, None), (15, None), (14, 50),
             (16, 64), (17, 100), (19, 2), (21, 0), (22, 0), (23, 0), (24, 8), (24, 3), (25, 0), (25, 70000)]
    for i, bad in cases:
        args = list(ok)
        args[i] = bad
        assert lib.plmc_cross_grad(*args) == -1, (i, bad)
    args = list(ok)
    args[12] = args[13] = args[15] = None            # no cotangent at all
    assert lib.plmc_cross_grad(*args) == -1
    args = list(ok)
    args[23], args[24] = 50, 52                      # wider than the kernel stages
    assert lib.plmc_cross_grad(*args) == -1
    assert lib.plmc_cross_grad_ws(256, 100, 3, 2) == 8 * 2 * 2 * 128 * 4
    for bad in ((200, 100, 3, 2), (256, 0, 3, 2), (256, 100, 0, 2), (256, 100, 3, 0)):
        assert lib.plmc_cross_grad_ws(*bad) == 0


def test_mix_tasks_bwd_rejects_bad_arguments():
    lib = _cabi.load()
    ok = [FAKE, FAKE, FAKE, FAKE, FAKE, 100, 100, 5, 2, None]
    for i, bad in [(2, None), (3, None), (4, None), (5, 50), (6, 0), (7, 0), (8, 0), (8, 70000)]:
        args = list(ok)
        args[i] = bad
        assert lib.plmc_mix_tasks_bwd(*args) == -1, (i, bad)
    args = list(ok)
    args[0] = args[1] = args[3] = args[4] = None
    assert lib.plmc_mix_tasks_bwd(*args) == -1


def test_sass_of_cross_grad_kernel_has_dmma():
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    sass = subprocess.run(["cuobjdump", "-sass", str(_cabi.lib_path())], capture_output=True, text=True).stdout
    seen = 0
    for block in sass.split("Function : ")[1:]:
        name = block.split("\n", 1)[0]
        if "cross_grad_kernel" in name:
            assert "DMMA.8x8x4" in block, name
            seen += 1
    assert seen == 20            # kernel ids 0-4 x four dimension widths
