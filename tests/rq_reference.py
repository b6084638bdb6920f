"""CPU reference of the rational quadratic kernel (gpytorch 1.11 RQKernel), built on the unchanged oracle.

gpytorch/kernels/rq_kernel.py: x / lengthscale, covar_dist(square_dist=True) -- the oracle's sq_dist, as for RBF --
then (1 + dist / (2 alpha)).pow(-alpha), alpha = softplus(raw_alpha) [q, 1] unsqueezed to [q, 1, 1].

The oracle evaluates every kernel through ``plmc_oracle.base_kernel``; ``rq_kernels(raw_alphas)`` puts an RQ-aware
version in its place for the duration of a block, so that ``gram``, ``mll``, ``predict``, the SGPR blocks and the joint
reference (tests/joint_reference.py) all evaluate RQ.  ``raw_alphas`` has one raw_alpha per additive component:
``gram`` visits the components in order, once each per call, and the i-th RQ evaluation of the block uses
``raw_alphas[i % len(raw_alphas)]``.  Params carry ``kernel="rq"``.
"""
import contextlib

import torch

from oracle import plmc_oracle as O


def rq_kernel(x1, x2, ell, zero_diag, alpha):
    """Batched ARD RQ kernel [q, n1, n2] for inputs [n, d], lengthscales [q, 1, d] and alpha (constrained) [q, 1]."""
    a = alpha.reshape(-1, 1, 1)
    return O.sq_dist(x1.div(ell), x2.div(ell), zero_diag).div(2 * a).add(1).pow(-a)


@contextlib.contextmanager
def rq_kernels(raw_alphas):
    base = O.base_kernel
    count = [0]

    def base_kernel(kind, x1, x2, ell, zero_diag):
        if kind != "rq":
            return base(kind, x1, x2, ell, zero_diag)
        raw = raw_alphas[count[0] % len(raw_alphas)]
        count[0] += 1
        return rq_kernel(x1, x2, ell, zero_diag, O.softplus(raw))

    O.base_kernel = base_kernel
    try:
        yield
    finally:
        O.base_kernel = base
