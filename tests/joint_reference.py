"""CPU references for the joint eval-mode posterior.  TEST INFRASTRUCTURE ONLY.

Built from the oracle's own pieces (oracle/plmc_oracle.py, oracle/kat.py), which stay as they are:
  predict_joint                 the projected form, along the lines of plmc_oracle.predict;
  dense_posterior_covariance    the same covariance through the dense multitask model (the KAT-2 construction of
                                oracle/kat.py with the full covariance instead of its diagonal).
"""
import torch

from oracle import kat
from oracle import plmc_oracle as O


def predict_joint(p: O.OracleParams, X: torch.Tensor, Y: torch.Tensor, Xs: torch.Tensor, max_tries: int = 3):
    """Joint predictive covariances of the exact GP.

    Returns (C [q, n*, n*], cov_f [N, N], cov_y [N, N]), N = n* p, point-major / task-minor: the latent posterior
    covariances C_l = K**_l - K*_l^T K_l^-1 K*_l, the covariance sum_l C_l (x) h_l h_l^T + eps I of the
    MultitaskMultivariateNormal the model returns (projected_lmc.py:1149-1155), and that covariance plus I (x) F F^T
    of the full likelihood.
    """
    n, ns = X.shape[0], Xs.shape[0]
    K = O.gram(p, X, training=False) + torch.diag_embed(O.noise(p)[:, None].expand(-1, n))
    L = O.psd_safe_cholesky(K, max_tries)
    Ks = O.gram(p, X, Xs, training=False)                                   # [q, n, n*]
    V = torch.linalg.solve_triangular(L, Ks, upper=False)
    C = O.gram(p, Xs, Xs, training=False) - V.transpose(-1, -2) @ V          # [q, n*, n*]
    Ht = O.lmc_coefficients(p)                                              # [q, p]
    ptasks = Ht.shape[1]
    cov_f = p.eps * torch.eye(ns * ptasks, dtype=X.dtype)
    for l in range(p.q):
        cov_f = cov_f + torch.kron(C[l], torch.outer(Ht[l], Ht[l]))
    Fch = O.task_noise_factor(p)
    cov_y = cov_f + torch.kron(torch.eye(ns, dtype=X.dtype), Fch @ Fch.T)
    return C, cov_f, cov_y


def dense_posterior_covariance(p: O.OracleParams, X: torch.Tensor, Y: torch.Tensor, Xs: torch.Tensor) -> torch.Tensor:
    """Posterior covariance of f at Xs (no noise, no eps) of the dense model, [n* p, n* p] point-major / task-minor."""
    n, ns = X.shape[0], Xs.shape[0]
    Ht = O.lmc_coefficients(p)
    ptasks = Ht.shape[1]
    C = kat.dense_task_covariance(p, X)
    Ks = O.gram(p, X, Xs, training=False)                  # [q, n, n*]
    Kss = O.gram(p, Xs, Xs, training=False)                # [q, n*, n*]
    cross = torch.zeros(n * ptasks, ns * ptasks, dtype=X.dtype)
    prior = torch.zeros(ns * ptasks, ns * ptasks, dtype=X.dtype)
    for l in range(p.q):
        hh = torch.outer(Ht[l], Ht[l])
        cross = cross + torch.kron(Ks[l], hh)
        prior = prior + torch.kron(Kss[l], hh)
    L = torch.linalg.cholesky(C)
    V = torch.linalg.solve_triangular(L, cross, upper=False)
    return prior - V.T @ V
