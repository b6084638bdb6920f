"""Timing of the joint posterior path (CUDA events after warm-up; needs one B200).

    python tools/joint_bench.py [--out profiles/r03_joint_bench.json]

C2 shape (n = 44 484, d = 21, q = 4, p = 7, Matern 5/2) at n* = 2048 and 4096: cross-Gram + V = L^-1 K*, the SYRK
V^T V (route and TFLOP/s-equivalent), K**, the task-covariance assembly (TB/s against the measured copy rate) and
log_prob of one value.  C4 per-GPU shape (n = 20 000, d = 8, q = 4, p = 500, RBF, n* = 1024): drawing S = 1000
samples through the latent structure, with the FLOP of a root of the dense covariance beside it.  FLOP and bytes are
algorithmic, computed from the shapes below.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile

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


def gemm_routes(fn):
    """Run fn with the per-GEMM trace on; return the trace report lines (the library prints them to stderr)."""
    ops.trace_enable(True)
    fn()
    torch.cuda.synchronize()
    with tempfile.TemporaryFile(mode="w+") as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            ops.trace_report()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        ops.trace_enable(False)
        f.seek(0)
        return [ln.split() for ln in f.read().splitlines()[1:] if ln.strip()]


def state(eng, n, d, q, kid, seed=0):
    g = torch.Generator().manual_seed(seed)
    dev = torch.device("cuda:0")
    X = (torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
    ell = torch.full((q, d), 0.8, dtype=torch.float64, device=dev)
    comps = [(kid, tuple(range(d)), ell, None)]
    TY = torch.randn(q, n, generator=g, dtype=torch.float64).to(dev)
    noise = torch.full((q,), 0.05, dtype=torch.float64, device=dev)
    st = eng.factorize(X, TY, comps, noise)
    return st, g


def c2(out, copy_rate):
    n, d, q, p, kid = 44484, 21, 4, 7, ops.KERNEL_IDS["matern52"]
    eng = LatentEngine()
    st, g = state(eng, n, d, q, kid)
    np_ = st["L"].shape[1]
    dev = st["L"].device
    H = torch.randn(q, p, generator=g, dtype=torch.float64).to(dev)
    S = 1e-3 * torch.eye(p, dtype=torch.float64, device=dev)
    res = []
    for ns in (2048, 4096):
        m = ops.npad(ns)
        Xs = (torch.rand(ns, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
        V = torch.empty((q, np_, m), dtype=torch.float64, device=dev)
        inverted = bool(st.get("inverted"))
        t_v = timeit(lambda: eng._cross_mean_v(st, Xs, V, m, inverted, True, zero_padding=True))
        lat_mean, C = eng.latent_covariance(st, Xs)
        C0 = C.clone()
        t_syrk = timeit(lambda: (C.copy_(C0), ops.syrk(V, C, -1.0, 1.0, eng.cfg_main)))
        t_copy = timeit(lambda: C.copy_(C0))
        t_syrk_only = max(t_syrk - t_copy, 1e-9)
        routes = gemm_routes(lambda: ops.syrk(V, C, -1.0, 1.0, eng.cfg_main))
        syrk_route = sorted({r[0] for r in routes if r[1:4] == [str(m), str(m), str(np_)]})
        Zs, zns = ops.scale_inputs(Xs, st["scaled"][0][3], st["comps"][0][2], m)
        zero = torch.zeros(q, dtype=torch.float64, device=dev)
        t_kss = timeit(lambda: ops.gram(Zs, zns, kid, None, zero, C, ns))
        N = ns * p
        t_task = timeit(lambda: ops.task_covariance(C0, H, S, ns))
        mean = torch.zeros(ns, p, dtype=torch.float64, device=dev)
        y = torch.randn(1, ns, p, generator=g, dtype=torch.float64).to(dev)
        with torch.no_grad():
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                t_lp = timeit(lambda: eng.joint_log_prob(C0, H, S, mean, y), reps=2)
        syrk_flop = q * m * m * np_                      # lower half of 2 m^2 npad per latent
        v_flop = q * float(n) * n * ns + 2.0 * q * n * ns * d * 3
        Np = ops.npad(N)
        res.append(dict(
            n_test=ns, m=m, N=N,
            cross_gram_and_V=dict(seconds=t_v, flop=v_flop, tflops=v_flop / t_v / 1e12,
                                  path="trmm by inv(L)" if inverted else "trsm"),
            syrk=dict(seconds=t_syrk_only, flop=syrk_flop, tflops_equiv=syrk_flop / t_syrk_only / 1e12,
                      route=syrk_route, shape=[m, m, np_, q]),
            k_star_star=dict(seconds=t_kss, bytes=8.0 * q * m * (m + 128) / 2,
                             tb_per_s=8.0 * q * m * (m + 128) / 2 / t_kss / 1e12),
            task_covariance_dense=dict(seconds=t_task, bytes=8.0 * N * N, flop=2.0 * q * N * N,
                                       tb_per_s=8.0 * N * N / t_task / 1e12,
                                       share_of_copy_rate=8.0 * N * N / t_task / copy_rate),
            log_prob_one_value=dict(seconds=t_lp, potrf_flop=Np ** 3 / 3.0, order=Np),
        ))
        del V, C, C0
        torch.cuda.empty_cache()
    out["c2"] = dict(n=n, d=d, q=q, p=p, kernel="matern52", results=res)


def c4(out):
    n, d, q, p, kid = 20000, 8, 4, 500, ops.KERNEL_IDS["rbf"]
    ns, S = 1024, 1000
    eng = LatentEngine()
    st, g = state(eng, n, d, q, kid, seed=1)
    dev = st["L"].device
    Xs = (torch.rand(ns, d, generator=g, dtype=torch.float64) * 2 - 1).to(dev)
    H = torch.randn(q, p, generator=g, dtype=torch.float64).to(dev)
    R = math.sqrt(1e-3) * torch.eye(p, dtype=torch.float64, device=dev)
    lat_mean, C = eng.latent_covariance(st, Xs)
    mean = torch.zeros(ns, p, dtype=torch.float64, device=dev)
    import warnings

    def draw():
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Lc, dinv = eng.factor_covariance(C, ns)
        eps = torch.randn((q, ns, S), dtype=torch.float64, device=dev)
        E = torch.randn((S, ns, p), dtype=torch.float64, device=dev)
        G = eng.latent_draws(Lc, dinv, eps)
        return ops.mix_samples(mean, G, H, E, R, ns, S)

    t = timeit(draw, reps=2)
    m = ops.npad(ns)
    latent_flop = q * m ** 3 / 3.0 + q * float(m) * m * S
    mix_flop = 2.0 * S * ns * p * (q + p)
    dense_flop = float(ns * p) ** 3 / 3.0
    out["c4_sampling"] = dict(n=n, d=d, q=q, p=p, n_test=ns, samples=S, seconds=t, latent_flop=latent_flop,
                              mix_flop=mix_flop, dense_root_flop=dense_flop,
                              bytes_written=8.0 * S * ns * p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "r03_joint_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("joint_bench.py measures on a GPU; none is available")
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    out = dict(device=torch.cuda.get_device_name(0), nvidia_smi=q[:1])
    src = torch.randn(1 << 28, dtype=torch.float64, device="cuda")       # 2 GiB: larger than L2
    dst = torch.empty_like(src)
    t = timeit(lambda: ops.peak_copy(src, dst))
    copy_rate = 16.0 * src.numel() / t
    out["copy_rate_tb_per_s"] = copy_rate / 1e12
    del src, dst
    c2(out, copy_rate)
    torch.cuda.empty_cache()
    c4(out)
    text = json.dumps(out, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
