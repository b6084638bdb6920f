"""Timing of the gradients of eval-mode predictions w.r.t. the test inputs (CUDA events, best of 3 after warm-up;
needs one B200).

    python tools/input_grad_bench.py [--out profiles/r05_input_grad_bench.json]

C2 shape (n = 44 484, d = 21, q = 4, p = 7, Matern 5/2) at n* = 2048 and 8192, one tile each:
  * the forward (LatentEngine.predict_latents: cross-Gram, latent means, V = L^-1 K*, variances);
  * the backward with mean-only cotangents (cross-Gram-free: one fused cross_grad sweep);
  * the backward with mean and variance cotangents (K*, then beta = L^-T L^-1 K*: two triangular products), with the
    factor L (trsm) and with the explicit inverse inv(L) (trmm);
  * cross_grad alone against the composed path: w materialised as the [q, n*, n] cotangent of the cross block with
    the test points as rows, then plmc_cross_gram_bwd2.
Analytic expectation: the variance backward costs about two triangular products per tile more than the forward
(2 q n^2 n* FLOP each way); the mean-only backward does no O(n^2 n*) work.  FLOP are algorithmic.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from projected_lmc_b200 import ops  # noqa: E402
from projected_lmc_b200.engine import LatentEngine  # noqa: E402


def timeit(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best / 1e3


def rel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "r05_input_grad_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("input_grad_bench.py measures on a GPU; none is available")
    torch.cuda.set_device(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi[:1])

    n, d, q, p, kid = 44484, 21, 4, 7, ops.KERNEL_IDS["matern52"]
    g = torch.Generator().manual_seed(0)
    dev = torch.device("cuda:0")
    X = (torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
    ell = torch.full((q, d), 0.8, dtype=torch.float64, device=dev)
    comps = [(kid, tuple(range(d)), ell, None)]
    TY = torch.randn(q, n, generator=g, dtype=torch.float64).to(dev)
    noise = torch.full((q,), 0.05, dtype=torch.float64, device=dev)
    eng = LatentEngine()
    eng.predict_inverse = False
    st = eng.factorize(X, TY, comps, noise)
    np_ = st["L"].shape[1]
    Z, zn = st["scaled"][0][0], st["scaled"][0][1]
    res = []
    tests = {}
    for ns in (2048, 8192):
        Xs = (torch.rand(ns, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
        gm = torch.randn(q, ns, generator=g, dtype=torch.float64).to(dev)
        gv = torch.randn(q, ns, generator=g, dtype=torch.float64).to(dev)
        tests[ns] = (Xs, gm, gv)
        r = dict(n_test=ns, tile=ns)
        r["forward_trsm_s"] = timeit(lambda: eng.predict_latents(st, Xs, tile=ns))
        r["backward_mean_only_s"] = timeit(lambda: eng.predict_latents_grad(st, Xs, gm, None, tile=ns))
        r["backward_mean_var_trsm_s"] = timeit(lambda: eng.predict_latents_grad(st, Xs, gm, gv, tile=ns))
        g_trsm = eng.predict_latents_grad(st, Xs, gm, gv, tile=ns)

        # the fused sweep alone against the composed adjoint, on the beta of this tile
        mt = ops.npad(ns)
        Zt, znt = ops.scale_inputs(Xs, st["scaled"][0][3], ell, mt)
        beta = torch.empty((q, np_, mt), dtype=torch.float64, device=dev)
        ops.cross_gram(Z, zn, Zt, znt, kid, None, beta, n, mt)
        ops.trsm(2, st["L"], st["dinv"], beta, 1.0, eng.cfg_main)
        ops.trsm(3, st["L"], st["dinv"], beta, 1.0, eng.cfg_main)
        alpha = st["alpha"]
        r["cross_grad_mean_var_s"] = timeit(lambda: ops.cross_grad(Z, zn, Zt, znt, kid, None, ell, alpha, n, ns, gm, gv,
                                                                   beta))
        r["cross_grad_mean_only_s"] = timeit(lambda: ops.cross_grad(Z, zn, Zt, znt, kid, None, ell, alpha, n, ns, gm))
        fused = ops.cross_grad(Z, zn, Zt, znt, kid, None, ell, alpha, n, ns, gm, gv, beta)
        G = torch.empty((q, ns, n), dtype=torch.float64, device=dev)

        def materialise():
            torch.mul(gm[:, :, None], alpha[:, None, :], out=G)
            G.add_(beta[:, :n, :ns].transpose(1, 2) * gv[:, :, None], alpha=-2.0)

        def composed():
            materialise()
            return ops.cross_gram_bwd(Zt, Z, G, kid, None, ell, ns, n)[2]

        r["composed_mean_var_s"] = timeit(composed)
        materialise()
        r["cross_gram_bwd2_alone_s"] = timeit(lambda: ops.cross_gram_bwd(Zt, Z, G, kid, None, ell, ns, n))
        r["fused_vs_composed_rel_err"] = rel(fused, composed())
        r["fused_speedup_over_composed"] = r["composed_mean_var_s"] / r["cross_grad_mean_var_s"]
        del G, beta
        torch.cuda.empty_cache()
        r["tri_flop_per_product"] = 2.0 * q * float(n) * n * ns / 2       # q n^2 n* (triangular)
        r["cross_grad_pairs"] = float(q) * n * ns
        r["_g_trsm"] = g_trsm
        res.append(r)

    # the same with the explicit inverse (trtri once per state, then trmm)
    eng.predict_inverse = True
    eng._maybe_invert(st, 1)
    for r in res:
        ns = r["n_test"]
        Xs, gm, gv = tests[ns]
        r["forward_trmm_s"] = timeit(lambda: eng.predict_latents(st, Xs, tile=ns))
        r["backward_mean_var_trmm_s"] = timeit(lambda: eng.predict_latents_grad(st, Xs, gm, gv, tile=ns))
        r["trmm_vs_trsm_grad_rel_err"] = rel(eng.predict_latents_grad(st, Xs, gm, gv, tile=ns), r.pop("_g_trsm"))
        r["backward_mean_var_over_forward_trsm"] = r["backward_mean_var_trsm_s"] / r["forward_trsm_s"]
        r["backward_mean_var_over_forward_trmm"] = r["backward_mean_var_trmm_s"] / r["forward_trmm_s"]
        r["backward_mean_only_over_forward_trsm"] = r["backward_mean_only_s"] / r["forward_trsm_s"]
    out["c2"] = dict(n=n, d=d, q=q, p=p, kernel="matern52", gemm_mode=eng.emulation_mode(), results=res)
    text = json.dumps(out, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
