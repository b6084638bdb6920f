"""Rational quadratic latent kernels next to RBF and Matern 5/2 (CUDA events after warm-up; needs one B200).

    python tools/rq_bench.py [--out profiles/r04_rq_bench.json] [--rounds 3]

1. Gram build and gradient sweep timed alone at n = 32 768, q = 4, d = 21 for RBF, Matern 5/2 and RQ in the same
   process, as a fraction of the device-to-device copy rate measured in the same run.  Bytes are algorithmic:
   8 q n (n + 1) / 2 written by the Gram, the same read by the sweep.  The working set (34 GB) is far above L2.
2. One full training iteration (forward + backward of the model's loss) at the C2 shape (n = 44 484, d = 21, p = 7,
   q = 4) with RQ and with Matern 5/2, alternated in the same process.  The engine of the kernel not being timed is
   released, and every timed iteration follows an untimed one of the same kernel.
"""
import argparse
import json
import os
import subprocess
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from projected_lmc_b200 import ProjectedGPModel, ProjectedLMCmll, gp, ops  # noqa: E402

KERNELS = {"rbf": (0, None), "matern52": (1, None), "rq": (4, 1.5)}


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def copy_rate(dev):
    n = 1 << 28                                   # 2 GB per buffer
    src = torch.ones(n, dtype=torch.float64, device=dev)
    dst = torch.empty_like(src)
    ms = min(events_ms(lambda: ops.peak_copy(src, dst), 5))
    return 16 * n / ms / 1e9                      # read + write bytes, TB/s


def kernel_alone(dev, rounds):
    n, q, d = 32768, 4, 21
    g = torch.Generator().manual_seed(0)
    X = (torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
    ell = torch.full((q, d), 0.9, dtype=torch.float64, device=dev)
    noise = torch.full((q,), 0.05, dtype=torch.float64, device=dev)
    np_ = ops.npad(n)
    Z, zn = ops.scale_inputs(X, ops.col_mean(X), ell, np_)
    K = torch.empty((q, np_, np_), dtype=torch.float64, device=dev)
    alpha = torch.randn(q, np_, generator=g, dtype=torch.float64).to(dev)
    nbytes = 8 * q * n * (n + 1) / 2
    res = {name: {"gram_ms": [], "sweep_ms": []} for name in KERNELS}
    for _ in range(rounds):                       # kernels alternated within every round
        for name, (kid, a) in KERNELS.items():
            shape = None if a is None else torch.full((q,), a, dtype=torch.float64, device=dev)
            res[name]["gram_ms"] += events_ms(lambda: ops.gram(Z, zn, kid, None, noise, K, n, shape=shape), 3)
            res[name]["sweep_ms"] += events_ms(lambda: ops.grad_sweep(K, alpha, Z, zn, ell, kid, None, n, shape=shape),
                                               3)
    out = {}
    for name, r in res.items():
        gm, sm = min(r["gram_ms"]), min(r["sweep_ms"])
        out[name] = dict(gram_ms=gm, sweep_ms=sm, gram_ms_all=r["gram_ms"], sweep_ms_all=r["sweep_ms"],
                         gram_tb_s=nbytes / gm / 1e9, sweep_tb_s=nbytes / sm / 1e9)
    return dict(n=n, q=q, d=d, bytes=nbytes, kernels=out)


def c2_iteration(dev, rounds):
    n, d, p, q = 44484, 21, 7, 4
    g = torch.Generator().manual_seed(1)
    X = torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1
    W = torch.randn(d, q, generator=g, dtype=torch.float64)
    Y = torch.sin(X @ W) @ torch.randn(q, p, generator=g, dtype=torch.float64) + 0.1 * torch.randn(n, p, generator=g)
    Y = (Y - Y.mean(0)) / Y.std(0)
    Xg, Yg = X.to(dev), Y.to(dev)
    models = {}
    for name, ktype in (("matern52", gp.kernels.MaternKernel), ("rq", gp.kernels.RQKernel)):
        torch.manual_seed(0)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m = ProjectedGPModel(X, Y, p, q, mean_type=gp.means.ZeroMean, kernel_type=ktype, BDN=False,
                                 init_lmc_coeffs=True).to(dev)
        with torch.no_grad():
            m._base_kernel().lengthscale = 1.5
        models[name] = m

    def step(m):
        m.zero_grad(set_to_none=True)
        loss = -ProjectedLMCmll(m.likelihood, m)(m(Xg), Yg)
        loss.backward()
        return loss

    times = {name: [] for name in models}
    losses = {}
    for _ in range(rounds):
        for name, m in models.items():
            for other in models.values():
                if other is not m:
                    other._engine.release()
            torch.cuda.empty_cache()
            step(m)                                 # untimed: workspace allocation and warm-up
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss = step(m)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
            losses[name] = loss.item()
    return dict(n=n, d=d, p=p, q=q, variant="PLMC", iteration_ms={k: v for k, v in times.items()},
                best_ms={k: min(v) for k, v in times.items()},
                rq_over_matern52=min(times["rq"]) / min(times["matern52"]), loss=losses)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r04_rq_bench.json")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rq_bench needs a CUDA device")
    torch.set_default_dtype(torch.float64)       # the model's parameters are created in the default dtype
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = dict(device=torch.cuda.get_device_name(dev), nvidia_smi=q[0] if q else None)
    res["copy_tb_s"] = copy_rate(dev)
    alone = kernel_alone(dev, args.rounds)
    for k in alone["kernels"].values():
        k["gram_of_copy"] = k["gram_tb_s"] / res["copy_tb_s"]
        k["sweep_of_copy"] = k["sweep_tb_s"] / res["copy_tb_s"]
    res["kernel_alone"] = alone
    torch.cuda.empty_cache()
    res["c2_iteration"] = c2_iteration(dev, args.rounds)
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
