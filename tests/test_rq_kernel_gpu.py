"""Rational quadratic latent kernels (gpytorch RQKernel) on the GPU: the Gram, cross-Gram and both gradient sweeps
(with the gradient of alpha) against the oracle / torch autograd, and the model paths (training, SGPR, prediction,
joint posterior, LOO, fp32, the INT8 routes, graphed fitting, jitter, device moves) against the CPU oracle."""
import warnings
from unittest import mock

import pytest
import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import ProjectedGPModel, ProjectedLMCmll, gp, ops
from projected_lmc_b200.engine import LatentEngine

from . import helpers
from .helpers import VARIANTS, cpu_copy, rel_err, synth
from .joint_reference import predict_joint
from .rq_reference import rq_kernel, rq_kernels

pytestmark = pytest.mark.gpu
DEV = "cuda"
MLL_TOL, GRAD_TOL, PRED_TOL = 1e-9, 1e-7, 1e-7


def inv_softplus(v):
    return v + torch.log(-torch.expm1(-v))


def make_rq_model(X, Y, q, variant="PLMC", outputscales=False, seed=0, **extra):
    torch.manual_seed(seed)
    kw = dict(VARIANTS[variant])
    kw.update(extra)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = ProjectedGPModel(X, Y, Y.shape[1], q, mean_type=gp.means.ZeroMean, kernel_type=gp.kernels.RQKernel,
                             init_lmc_coeffs=True, outputscales=outputscales, **kw)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():          # off the symmetric init, so that every gradient path is exercised
        for name, prm in m.named_parameters():
            if "Q_plus" not in name:
                prm.add_(0.1 * torch.randn(prm.shape, generator=g, dtype=prm.dtype))
    return m


def rq_oracle_params(mc):
    """helpers.oracle_params with the RQ kernel's name, and the raw_alpha of every component in order (for
    rq_reference.rq_kernels)."""
    with mock.patch.dict(helpers.KNAMES, {4: "rq"}):
        p = helpers.oracle_params(mc)
    cov = mc._covar()
    kers = list(cov.kernels) if hasattr(cov, "kernels") else [cov]
    return p, [(k.base_kernel if hasattr(k, "base_kernel") else k).raw_alpha for k in kers]


# ---- kernel level -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,with_os", [(100, 1, False), (300, 6, True), (257, 21, False)])
def test_rq_gram_and_cross_gram_vs_oracle(n, d, with_os):
    q = 3
    g = torch.Generator().manual_seed(n + d)
    X = torch.rand(n, d, generator=g) * 2 - 1
    ell = torch.rand(q, d, generator=g) + 0.4
    noise = torch.rand(q, generator=g) * 0.3 + 0.05
    alpha = torch.tensor([0.05, 1.3, 40.0])
    os_ = (torch.rand(q, generator=g) + 0.5) if with_os else None
    Xg = X.to(DEV)
    osg = None if os_ is None else os_.to(DEV)
    np_ = ops.npad(n)
    Z, zn = ops.scale_inputs(Xg, ops.col_mean(Xg), ell.to(DEV), np_)
    K = torch.full((q, np_, np_), float("nan"), dtype=torch.float64, device=DEV)
    ops.gram(Z, zn, ops.KERNEL_RQ, osg, noise.to(DEV), K, n, shape=alpha.to(DEV))
    p = O.OracleParams(raw_lengthscale=inv_softplus(ell)[:, None, :], raw_noise=inv_softplus(noise)[:, None],
                       noise_lower=0.0, kernel="rq", raw_outputscale=None if os_ is None else inv_softplus(os_))
    raw_alphas = [inv_softplus(alpha)[:, None]]
    with rq_kernels(raw_alphas):
        Kref = O.gram(p, X, training=False) + torch.diag_embed(noise[:, None].expand(-1, n))
    low = torch.tril(torch.ones(n, n, dtype=torch.bool))
    assert (K[:, :n, :n].cpu() - Kref)[:, low].abs().max().item() < 1e-12
    ns = 150
    Xs = torch.rand(ns, d, generator=g) * 2 - 1
    mt = ops.npad(ns)
    Zt, znt = ops.scale_inputs(Xs.to(DEV), ops.col_mean(Xg), ell.to(DEV), mt)
    Kx = torch.empty((q, np_, mt), dtype=torch.float64, device=DEV)
    ops.cross_gram(Z, zn, Zt, znt, ops.KERNEL_RQ, osg, Kx, n, mt, shape=alpha.to(DEV))
    with rq_kernels(raw_alphas):
        Kxref = O.gram(p, X, Xs, training=False)
    assert (Kx[:, :n, :ns].cpu() - Kxref).abs().max().item() < 1e-12
    with pytest.raises(ops.PlmcError):
        ops.gram(Z, zn, ops.KERNEL_RQ, osg, noise.to(DEV), K, n)


@pytest.mark.parametrize("n,d,with_os", [(300, 3, True), (257, 21, False), (150, 30, True)])
def test_rq_sweep_vs_autograd(n, d, with_os):
    """Both sweeps (GEMM form for d <= 24, direct differences for any d) against autograd of
    f = sum_ij W_ij K_ij, W = 1/2 (a a^T - Kinv) held fixed, including d f / d alpha."""
    q = 2
    g = torch.Generator().manual_seed(n * 31 + d)
    X = torch.rand(n, d, generator=g) * 2 - 1
    ell = (torch.rand(q, d, generator=g) + 0.4).requires_grad_(True)
    alpha = torch.tensor([0.3, 7.0], requires_grad=True)
    os_ = (torch.rand(q, generator=g) + 0.5).requires_grad_(True) if with_os else None
    a = torch.randn(q, n, generator=g)
    M = torch.randn(q, n, n, generator=g)
    Kinv = M @ M.transpose(1, 2) / n
    W = 0.5 * (a[:, :, None] * a[:, None, :] - Kinv)
    f = torch.zeros(())
    for l in range(q):
        Kl = rq_kernel(X, X, ell[l:l + 1], zero_diag=True, alpha=alpha[l:l + 1])
        f = f + (W[l] * (Kl if os_ is None else os_[l] * Kl)).sum()
    f.backward()
    np_ = ops.npad(n)
    Xg = X.to(DEV)
    Z, zn = ops.scale_inputs(Xg, ops.col_mean(Xg), ell.detach().to(DEV), np_)
    Kp = torch.eye(np_, dtype=torch.float64, device=DEV).repeat(q, 1, 1)
    Kp[:, :n, :n] = torch.tril(Kinv).to(DEV) + torch.triu(torch.full((n, n), float("nan")), 1).to(DEV)
    ap = torch.zeros((q, np_), dtype=torch.float64, device=DEV)
    ap[:, :n] = a.to(DEV)
    osg = None if os_ is None else os_.detach().to(DEV)
    try:
        for direct in (False, True):
            ops.sweep_debug(direct)
            g_ell, g_os, g_noise, g_alpha = ops.grad_sweep(Kp, ap, Z, zn, ell.detach().to(DEV), ops.KERNEL_RQ, osg, n,
                                                           shape=alpha.detach().to(DEV))
            assert rel_err(g_ell, ell.grad) < 1e-10, direct
            assert rel_err(g_alpha, alpha.grad) < 1e-10, (direct, g_alpha.cpu(), alpha.grad)
            assert rel_err(g_noise, torch.diagonal(W, dim1=1, dim2=2).sum(-1)) < 1e-12, direct
            if os_ is not None:
                assert rel_err(g_os, os_.grad) < 1e-11, direct
    finally:
        ops.sweep_debug(False)


@pytest.mark.parametrize("d", [3, 21, 30])
def test_old_and_new_entry_points_are_bit_identical_for_kernels_0_to_3(d):
    n, q = 600, 2
    g = torch.Generator().manual_seed(d)
    X = (torch.rand(n, d, generator=g) * 2 - 1).to(DEV)
    ell = (torch.rand(q, d, generator=g) + 0.4).to(DEV)
    os_ = (torch.rand(q, generator=g) + 0.5).to(DEV)
    noise = torch.full((q,), 0.1, dtype=torch.float64, device=DEV)
    np_ = ops.npad(n)
    Z, zn = ops.scale_inputs(X, ops.col_mean(X), ell, np_)
    lib = ops.lib()
    P = ops.ptr
    dp = Z.shape[2]
    a = torch.randn(q, np_, generator=g).to(DEV)
    for kid in range(4):
        K1 = torch.zeros((q, np_, np_), dtype=torch.float64, device=DEV)
        K2 = torch.zeros_like(K1)
        assert lib.plmc_gram(P(Z), P(zn), kid, P(os_), P(noise), P(K1), np_, np_ * np_, n, np_, dp, q, 0,
                             ops.stream()) == 0
        assert lib.plmc_gram2(P(Z), P(zn), kid, P(os_), None, P(noise), P(K2), np_, np_ * np_, n, np_, dp, q, 0,
                              ops.stream()) == 0
        assert torch.equal(K1, K2)
        outs = []
        for new in (False, True):
            ws = torch.zeros(lib.plmc_grad_ws(np_, d, q) // 8, dtype=torch.float64, device=DEV)
            ge, go, gn = (torch.zeros(q, d, dtype=torch.float64, device=DEV), torch.zeros(q, dtype=torch.float64, device=DEV),
                          torch.zeros(q, dtype=torch.float64, device=DEV))
            if new:
                rc = lib.plmc_grad_sweep2(P(K1), np_, np_ * np_, P(a), np_, P(Z), P(zn), P(ell), kid, P(os_), None,
                                          P(ge), P(go), P(gn), None, P(ws), n, np_, d, dp, q, ops.stream())
            else:
                rc = lib.plmc_grad_sweep(P(K1), np_, np_ * np_, P(a), np_, P(Z), P(zn), P(ell), kid, P(os_), P(ge),
                                         P(go), P(gn), P(ws), n, np_, d, dp, q, ops.stream())
            assert rc == 0
            outs.append((ge, go, gn))
        for x, y in zip(*outs):
            assert torch.equal(x, y)


# ---- model level ------------------------------------------------------------------------------------------------
def run_rq_case(n, d, p, q, variant, outputscales=False, ns=37, seed=0, mll_tol=MLL_TOL, grad_tol=GRAD_TOL,
                pred_tol=PRED_TOL, m=None, X=None, Y=None, Xs=None, **model_kwargs):
    if m is None:
        X, Y, Xs, _ = synth(n, d, p, q, seed=seed, ns=ns)
        m = make_rq_model(X, Y, q, variant=variant, outputscales=outputscales, seed=seed, **model_kwargs)
    mc = cpu_copy(m)
    m = m.cuda()
    m.train()
    loss = -ProjectedLMCmll(m.likelihood, m)(m(X.cuda()), Y.cuda())
    loss.backward()
    mc.train()
    p, raw_alphas = rq_oracle_params(mc)
    with rq_kernels(raw_alphas):
        ref = -O.mll(p, X, Y)
    ref.backward()
    assert abs(loss.item() - ref.item()) <= mll_tol * abs(ref.item()), (loss.item(), ref.item())
    ref_grads = dict(mc.named_parameters())
    seen_alpha = False
    for name, prm in m.named_parameters():
        g_ref = ref_grads[name].grad
        if g_ref is None:
            assert prm.grad is None or prm.grad.abs().max().item() == 0.0, name
            continue
        seen_alpha |= name.endswith("raw_alpha")
        assert rel_err(prm.grad, g_ref) <= grad_tol, (name, prm.grad.cpu(), g_ref)
    assert seen_alpha
    m.eval()
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        lat = m(Xs.cuda())
        obs = m.full_likelihood()(lat)
        p, raw_alphas = rq_oracle_params(mc)
        with rq_kernels(raw_alphas):
            mean_ref, varf_ref, vary_ref = O.predict(p, X, Y, Xs)
    assert rel_err(lat.mean, mean_ref) <= pred_tol
    assert rel_err(lat.variance, varf_ref) <= pred_tol
    assert rel_err(obs.variance, vary_ref) <= pred_tol
    return m, mc


@pytest.mark.parametrize("variant", ["PLMC", "PLMC_fast", "BDN_full"])
@pytest.mark.parametrize("outputscales", [False, True])
def test_rq_model_vs_oracle(variant, outputscales):
    run_rq_case(n=150, d=3, p=7, q=3, variant=variant, outputscales=outputscales)


def test_rq_decomp_with_lengthscale_priors():
    run_rq_case(n=140, d=4, p=6, q=2, variant="PLMC", decomp=[[0, 1], [1, 2, 3]],
                prior_scales=torch.tensor([0.8, 1.1, 0.9, 1.3]), prior_width=torch.tensor([0.5, 0.3, 0.4, 0.2]))


def test_rq_sgpr_vs_oracle():
    run_rq_case(n=300, d=3, p=5, q=2, variant="PLMC", n_inducing_points=40, mll_tol=1e-8, grad_tol=1e-6,
                pred_tol=1e-6)


def test_rq_joint_posterior_loo_and_cond():
    X, Y, Xs, _ = synth(160, 3, 5, 2, seed=3, ns=30)
    m = make_rq_model(X, Y, 2, variant="PLMC", outputscales=True, seed=3)
    mc = cpu_copy(m)
    m = m.cuda().eval()
    op, raw_alphas = rq_oracle_params(mc)
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pred = m(Xs.cuda())
        with rq_kernels(raw_alphas):
            C, cov_f, _ = predict_joint(op, X, Y, Xs)
        assert rel_err(pred.covariance_matrix, cov_f) < PRED_TOL
        lp = pred.log_prob(Y[:30].cuda())
        ref = torch.distributions.MultivariateNormal(pred.mean.cpu().reshape(-1), cov_f).log_prob(Y[:30].reshape(-1))
        assert abs(lp.item() - ref.item()) <= PRED_TOL * abs(ref.item())
        s2, r = m.compute_loo()
        with rq_kernels(raw_alphas):
            K = O.gram(op, X, training=False) + torch.diag_embed(O.noise(op)[:, None].expand(-1, 160))
        Kinv = torch.linalg.inv(K)
        s2_ref = 1.0 / torch.diagonal(Kinv, dim1=1, dim2=2)
        r_ref = (Kinv @ O.project_data(op, Y).unsqueeze(-1)).squeeze(-1) * s2_ref
        assert rel_err(s2, s2_ref.T) < 1e-8 and rel_err(r, r_ref.T) < 1e-8
        assert rel_err(m.kernel_cond(), torch.linalg.cond(K)) < 1e-8


def test_rq_fp32_grade():
    X, Y, Xs, _ = synth(200, 3, 5, 2, seed=5, ns=20)
    m = make_rq_model(X, Y, 2, variant="PLMC", seed=5)
    mc = cpu_copy(m)
    m32 = m.float().cuda()
    loss = -ProjectedLMCmll(m32.likelihood, m32)(m32(X.float().cuda()), Y.float().cuda())
    loss.backward()
    p, raw_alphas = rq_oracle_params(mc)
    with rq_kernels(raw_alphas):
        ref = -O.mll(p, X, Y)
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 1e-4 * abs(ref.item())
    refg = dict(mc.named_parameters())
    for name, prm in m32.named_parameters():
        if refg[name].grad is not None:
            assert rel_err(prm.grad, refg[name].grad) < 1e-4, name


def test_rq_int8_routes_agree():
    """n = 2600: the factorisation layer takes the INT8 tensor path; residues, digit planes and pure FP64 agree."""
    X, Y, _, _ = synth(2600, 4, 5, 2, seed=7)
    res = {}
    old = LatentEngine.gemm_mode
    try:
        for mode in ("rns", "digits", "fp64"):
            LatentEngine.gemm_mode = mode
            m = make_rq_model(X, Y, 2, variant="PLMC", seed=7).cuda()
            m._engine.rns_min_mnk = int(1e9)
            loss = -ProjectedLMCmll(m.likelihood, m)(m(X.cuda()), Y.cuda())
            loss.backward()
            res[mode] = (loss.item(), {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None})
            assert m._engine.emulation_mode() == mode
    finally:
        LatentEngine.gemm_mode = old
    for mode in ("rns", "digits"):
        assert abs(res[mode][0] - res["fp64"][0]) <= 1e-9 * abs(res["fp64"][0])
        for k, g in res["fp64"][1].items():
            assert rel_err(res[mode][1][k], g) < 1e-9, (mode, k)


def test_rq_fit_with_cuda_graphs_follows_the_eager_loop():
    from projected_lmc_b200 import fit

    X, Y, _, _ = synth(300, 3, 6, 2, seed=11)
    outs, finals, alphas = {}, {}, {}
    for mode in (False, True):
        m = make_rq_model(X, Y, 2, variant="PLMC", seed=11).cuda()
        a0 = m._base_kernel().alpha.detach().clone()
        outs[mode] = fit(m, ProjectedLMCmll(m.likelihood, m), m.train_inputs[0], m.train_y, n_iter=8, lr=1e-2,
                         lr_min=1e-3, check_every=4, cuda_graph=mode)
        finals[mode] = [p.detach().cpu().clone() for p in m.parameters()]
        alphas[mode] = (a0, m._base_kernel().alpha.detach().clone())
    assert outs[True]["cuda_graph"], outs[True]["cuda_graph_note"]
    assert not torch.equal(*alphas[True])          # alpha moved: the static copy was refreshed before each replay
    assert rel_err(outs[True]["losses"], outs[False]["losses"]) < 1e-10
    for a, b in zip(finals[True], finals[False]):
        assert rel_err(a, b) < 1e-7


def test_rq_jitter_retry_on_duplicated_points():
    # duplicate points + tiny noise on latent 0: its first factorisation fails, jitter goes to that latent only
    X, Y, _, _ = synth(120, 2, 5, 2, seed=13)
    X[60:] = X[:60]
    m = make_rq_model(X, Y, 2, variant="PLMC_fast", seed=13, noise_thresh=-40.0)
    with torch.no_grad():
        m.likelihood.noise_covar.raw_noise[0] = -60.0
        m._base_kernel().raw_lengthscale.fill_(0.5)
    mc = cpu_copy(m)
    m = m.cuda()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with gp.settings.cholesky_max_tries(8):
            val = ProjectedLMCmll(m.likelihood, m)(m(X.cuda()), Y.cuda()).item()
        p, raw_alphas = rq_oracle_params(mc)
        with rq_kernels(raw_alphas):
            ref = O.mll(p, X, Y, max_tries=8).item()
    assert m._engine.last_jitter is not None and m._engine.last_jitter[1].item() == 0.0
    assert abs(val - ref) <= 1e-6 * abs(ref)


def test_rq_state_dict_round_trip_through_cuda():
    X, Y, Xs, _ = synth(120, 3, 5, 2, seed=17, ns=10)
    m = make_rq_model(X, Y, 2, variant="PLMC", outputscales=True, seed=17)
    m._base_kernel().alpha = torch.tensor([[0.4], [5.0]])
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    mg = make_rq_model(X, Y, 2, variant="PLMC", outputscales=True, seed=99).cuda()
    mg.load_state_dict({k: v.cuda() for k, v in sd.items()})
    assert torch.equal(mg._base_kernel().raw_alpha.cpu(), sd["covar_module.base_kernel.raw_alpha"])
    back = {k: v.cpu() for k, v in mg.state_dict().items()}
    assert all(torch.equal(back[k], sd[k]) for k in sd)
    mg.eval()
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        mean = mg(Xs.cuda()).mean
        p, raw_alphas = rq_oracle_params(cpu_copy(mg).cpu())
        with rq_kernels(raw_alphas):
            mean_ref, _, _ = O.predict(p, X, Y, Xs)
    assert rel_err(mean, mean_ref) < PRED_TOL
