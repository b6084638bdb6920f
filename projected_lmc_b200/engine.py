"""Device-side orchestration of the latent-GP computations (one instance per model).

This is the Python host side above the C ABI: it owns the (cached) HBM workspaces
and sequences the stream-ordered kernels of csrc/ for
  * training:  scale -> Gram -> potrf (jitter retry) -> solve/logdet -> potri -> fused sweep
  * prediction: factorise once per parameter state, then tile the test points.
It contains no numerical fallback: every array operation on the O(n^2)/O(n^3)
path is a libplmc_b200 kernel.

HBM layout (per model, q_local latents of order n, npad = ceil(n/128)*128):
  K     [q, npad, npad]  f64  Gram -> L -> L^-1 -> K^-1, all in place (lower 128-tiles)
  dinv  [q, npad/128, 128, 128] f64  inverses of the diagonal leaves of L
  rhs   [q, npad, 128]   f64  right-hand-side panel of the two triangular solves
  Z     [q, npad, dpad]  f64  centred inputs divided by the lengthscales; zn [q, npad]
"""
from __future__ import annotations

import contextlib
import gc
import math
import warnings

import torch

from . import ops
from ._cabi import PlmcError, npad as _npad
from .gp import settings


@contextlib.contextmanager
def no_gc_during_capture():
    """A cyclic garbage collection that runs while a stream is capturing can destroy an unrelated CUDA graph or
    free memory of its private pool -- cudaFree / cudaGraphExecDestroy are not allowed then, and the failure is raised
    inside a destructor (the process aborts).  torch.cuda.graph() collects once BEFORE the capture starts; with the
    collector switched off for the duration of the capture nothing is destroyed in the middle of it."""
    was = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if was:
            gc.enable()


class NotPSDError(RuntimeError):
    pass


class NanError(RuntimeError):
    """Raised where linear_operator's psd_safe_cholesky raises its NanError (NaN in the matrix to factor)."""


class LatentEngine:
    """Per-model device orchestration.  All numerical settings travel with each library call (plmc_gemm_cfg);
    nothing here touches process-wide state, so engines with different settings may run concurrently on
    different streams or devices."""

    def __init__(self):
        self._ws = None
        self._ws_key = None
        self._xmean = None
        self._xmean_key = None
        self._oz = None
        self._cfg = (None, None)
        self._cfg_key = None
        self._pinned = None
        self._force_eager = False
        self._xsub = {}
        self._graphs = {}
        self.last_jitter = None
        self.generation = 0     # bumped whenever ws['K'] is rewritten (prediction caches compare it)

    # -- workspaces -----------------------------------------------------------
    def workspace(self, device, q: int, n: int):
        np_ = _npad(n)
        key = (str(device), q, np_)
        if self._ws_key != key:
            self._ws = None  # release before re-allocating
            self._ws = dict(
                K=torch.empty((q, np_, np_), dtype=torch.float64, device=device),
                dinv=ops.alloc_dinv(np_, q, device),
                rhs=torch.empty((q, np_, 128), dtype=torch.float64, device=device),
                info=torch.zeros((q + 1,), dtype=torch.int32, device=device),   # [q] = non-finite-input flag
            )
            self._ws_key = key
            self._oz, self._cfg_key = None, None
            self._graphs = {}
        self._configure_fp64(device, np_, q)
        return self._ws

    # -- FP64 through the INT8 tensor path for the large GEMMs ----------------------------------------
    # gemm_mode: "rns"    residue planes (csrc/ozaki2.cu): rns_moduli INT8 products per FP64 product
    #                     (16 = 55 operand bits for K <= 16384, DGEMM-grade; 14 = 47 bits);
    #            "digits" 8-bit digit planes (csrc/ozaki.cu): fp64_slices planes, s(s+1)/2 products
    #                     (7 = 55 bits, 6 = 47 bits);
    #            "fp64"   pure DMMA arithmetic (also selected by fp64_slices = 0 / PLMC_FP64_SLICES=0).
    # fp64_min_dim: smallest GEMM dimension routed to the INT8 path.  Defaults come from the environment so
    # that the whole test-suite can be run in any mode.
    gemm_mode = __import__("os").environ.get("PLMC_GEMM_MODE", "rns")
    fp64_slices = int(__import__("os").environ.get("PLMC_FP64_SLICES", "7"))
    fp64_min_dim = int(__import__("os").environ.get("PLMC_FP64_MIN_DIM", "128"))
    # ... and the least work M*N*K (default 512^3: with min_dim 128 the tall-skinny m x 128 x 128 leaf applications
    # of the triangular solves take the tensor path from m = 8192 on, the small products stay on DMMA)
    fp64_min_mnk = int(float(__import__("os").environ.get("PLMC_FP64_MIN_MNK", str(512 ** 3))))
    fp64_min_order = 1024    # matrices below this order are factorised in pure FP64
    # CUDA-graph replay of the engine part of a training step (launch-bound problems such as BASELINE config 1:
    # ~130 library launches per iteration at n = 1000 become two graph launches).  Matrices of order <= this are
    # captured after one eager warm-up call; 0 switches it off.
    graph_max_order = int(__import__("os").environ.get("PLMC_GRAPH_MAX_ORDER", "4096"))
    capture_mode = False     # True while training.fit captures / replays the WHOLE step as a CUDA graph
    capture_info = None
    max_sweep_dims = 44      # csrc/gram.cu grad_sweep_kernel: (2*128*(dpad+1) + ...)*8 bytes <= 227 KB
    # Moduli of the residue-plane products.  The whole O(n^3) layer runs power-capped with the INT8 pipe saturated
    # (DESIGN.md section 3.7: ~2.0 POPS at ~850 MHz under the 1000 W cap), so its time is proportional to the number
    # of INT8 products per FP64 product, i.e. to these two numbers.
    # Factorisation, solves, prediction: 15 moduli = 50-53 operand bits (plmc_rns_bits), a DGEMM's own rounding level:
    # at n = 20000, cond ~ 1e8 the loss moves by 6e-13 and the gradients by 4e-11 against 16 moduli, while pure FP64
    # DMMA arithmetic itself sits 9e-13 / 8e-10 away (tools/kinv_scale_check.py, profiles/r02_moduli_at_scale.jsonl);
    # tolerances 1e-8 / 1e-6.
    rns_moduli = int(__import__("os").environ.get("PLMC_RNS_MODULI", "15"))
    # Explicit inverse of the training iteration (K^-1 = L^-T L^-1: trtri + lauum).  K^-1 feeds ONLY the gradient
    # sweep tr((alpha alpha^T - K^-1) dK): the loss, alpha and the log-determinant come from L.  12 moduli = 39-42
    # bits: in the same measurement the gradients move by 4e-12 between 16, 13, 12 and even 11 moduli -- two orders
    # below the FP64-vs-INT8 difference, five below the tolerance.  0 = same as the main one.
    fp64_slices_kinv = int(__import__("os").environ.get("PLMC_FP64_SLICES_KINV", "6"))
    rns_moduli_kinv = int(__import__("os").environ.get("PLMC_RNS_MODULI_KINV", "12"))
    # fp32 grade (models whose tensors are float32; the reference's GPU default, experiments.py:4-8, tolerance 1e-4):
    # storage and accumulation stay FP64, but the operands of the large products carry 32 bits (10 moduli =
    # 10 INT8 products, or 4 digit planes = 10 products) in the factorisation AND the inverse: a third fewer
    # tensor operations than the fp64 grade, results ~1e-8 from the FP64 ones (far inside 1e-4)
    grade = "fp64"
    rns_moduli_f32 = int(__import__("os").environ.get("PLMC_RNS_MODULI_F32", "10"))
    fp64_slices_f32 = int(__import__("os").environ.get("PLMC_FP64_SLICES_F32", "4"))
    rns_flags = int(__import__("os").environ.get("PLMC_RNS_FLAGS", "0"))
    # the residue scheme pays a fixed cost per output element: products with K < rns_min_k or M*N*K < rns_min_mnk
    # run on digit planes of the matching grade (fp64_slices / fp64_slices_kinv) instead; 0 = residues everywhere
    rns_min_k = int(__import__("os").environ.get("PLMC_RNS_MIN_K", "1024"))
    rns_min_mnk = int(float(__import__("os").environ.get("PLMC_RNS_MIN_MNK", "2e10")))
    scratch_cap_bytes = int(float(__import__("os").environ.get("PLMC_SCRATCH_GB", "48")) * (1 << 30))

    def emulation_mode(self):
        if self.fp64_slices <= 0 or self.gemm_mode == "fp64":
            return "fp64"
        return "rns" if self.gemm_mode == "rns" else "digits"

    def _configure_fp64(self, device, np_, q=1):
        mode, md = self.emulation_mode(), self.fp64_min_dim
        f32 = (self.grade == "fp32")
        key = (mode, f32, md, self.fp64_min_mnk, self.fp64_slices, self.fp64_slices_kinv, self.rns_moduli, self.rns_moduli_kinv,
               self.rns_flags, self.rns_min_k, self.rns_min_mnk, str(device), np_, q)
        if key == self._cfg_key:
            return
        self._cfg_key = key
        if mode == "fp64" or np_ < max(self.fp64_min_order, 2 * md):
            self._cfg = (None, None)
            return
        h = np_ // 2
        if mode == "rns":
            # planes + residue tiles of the largest product of the recursion (the top-level SYRK) per latent;
            # a product that does not fit is split inside the library, batch members are processed in passes
            m = self.rns_moduli
            per_member = max(m * h * h + m * (h + 256) * (h + 256) // 2 + m * h * 8192,
                             self.fp64_slices * h * (h + 8192)) + (1 << 20)
        else:
            # digit planes of the largest GEMM (s * (M + N) * K bytes, M, K <= npad/2, N <= npad/2 or a
            # prediction tile); a GEMM whose planes do not fit falls back to the DMMA kernel
            per_member = self.fp64_slices * h * (h + 8192) + (1 << 20)
        cap = self.scratch_cap_bytes
        if device.type == "cuda":
            free, _ = torch.cuda.mem_get_info(device)
            have = self._oz.numel() if self._oz is not None and self._oz.device == device else 0
            cap = max(per_member // 8, min(cap, free + have - (6 << 30)))
        need = int(min(q * per_member, max(cap, 1 << 26)))
        if self._oz is None or self._oz.numel() < need or self._oz.device != device:
            self._oz = None
            self._oz = torch.empty((need,), dtype=torch.uint8, device=device)
        if mode == "rns":
            mm = min(self.rns_moduli_f32, self.rns_moduli) if f32 else self.rns_moduli
            mk = mm if f32 else min(self.rns_moduli_kinv or self.rns_moduli, self.rns_moduli)
            sl = min(self.fp64_slices_f32, self.fp64_slices) if f32 else self.fp64_slices
            alt = sl if (self.rns_min_k > 0 or self.rns_min_mnk > 0) else 0
            altk = alt if f32 else min(self.fp64_slices_kinv or alt, alt)
            self._cfg = (ops.gemm_cfg(self._oz, ops.GEMM_INT8_RNS, mm, md, self.rns_flags, alt,
                                      self.rns_min_k, self.rns_min_mnk, self.fp64_min_mnk),
                         ops.gemm_cfg(self._oz, ops.GEMM_INT8_RNS, mk, md, self.rns_flags, altk,
                                      self.rns_min_k, self.rns_min_mnk, self.fp64_min_mnk))
        else:
            sm_ = min(self.fp64_slices_f32, self.fp64_slices) if f32 else self.fp64_slices
            sk = sm_ if f32 else min(self.fp64_slices_kinv or self.fp64_slices, self.fp64_slices)
            self._cfg = (ops.gemm_cfg(self._oz, ops.GEMM_INT8_DIGITS, sm_, md, min_mnk=self.fp64_min_mnk),
                         ops.gemm_cfg(self._oz, ops.GEMM_INT8_DIGITS, sk, md, min_mnk=self.fp64_min_mnk))

    @property
    def cfg_main(self):
        return self._cfg[0]

    @property
    def cfg_kinv(self):
        return self._cfg[1]

    def release(self):
        """Drop the HBM workspaces and the plane scratch."""
        self._graphs = {}
        self._ws, self._ws_key = None, None
        self._oz, self._cfg, self._cfg_key = None, (None, None), None

    def xmean(self, X: torch.Tensor) -> torch.Tensor:
        key = (X.data_ptr(), X._version, tuple(X.shape), str(X.device))
        if self._xmean_key != key:
            self._xmean = ops.col_mean(X)
            self._xmean_key = key
            self._xsub = {}
        return self._xmean

    def _forget_inputs(self):
        """Drops what was derived from the contents of the inputs (column means, per-component input subsets)."""
        self._xmean_key, self._xsub = None, {}

    def _sub_inputs(self, X, dims):
        """(X[:, dims] contiguous, its column means) for one component of an additive kernel (cached with X)."""
        full = self.xmean(X)
        if tuple(dims) == tuple(range(X.shape[1])):
            return X, full
        hit = self._xsub.get(tuple(dims))
        if hit is None:
            idx = torch.as_tensor(list(dims), device=X.device)
            Xg = X.index_select(1, idx).contiguous()
            hit = (Xg, ops.col_mean(Xg))
            self._xsub[tuple(dims)] = hit
        return hit

    def _scaled(self, X, comps, rows_pad):
        """Per component: (Z [q, rows_pad, dpad_g], zn, X_g, xmean_g)."""
        out = []
        for kid, dims, ell, os_ in comps:
            if len(dims) > self.max_sweep_dims:
                # the gradient sweep stages full-width scaled inputs of both tile sides in shared memory
                raise PlmcError(f"a kernel over {len(dims)} input dimensions exceeds the {self.max_sweep_dims} the "
                                "gradient sweep stages in shared memory; split it with `decomp` into additive groups")
            Xg, xm = self._sub_inputs(X, dims)
            Z, zn = ops.scale_inputs(Xg, xm, ell, rows_pad)
            out.append((Z, zn, Xg, xm))
        return out

    @staticmethod
    def _gram_all(comps, scaled, diag_add, K, n, sl=None):
        """K = sum_g os_g k_g + diag_add I (lower tiles, identity padding); sl restricts to a slice of latents."""
        for g, (c, (Z, zn, _, _)) in enumerate(zip(comps, scaled)):
            kid, dims, ell, os_ = c
            shape = ops.shape_of(c)
            if sl is not None:
                Z, zn = Z[sl], zn[sl]
                os_ = None if os_ is None else os_[sl]
                shape = None if shape is None else shape[sl]
            ops.gram(Z, zn, kid, os_, diag_add, K, n, accumulate=(g > 0), shape=shape)

    # -- factorisation with gpytorch's psd_safe_cholesky retry semantics ---------
    # The first attempt is launched WITHOUT a host synchronisation: `info` (first bad pivot per latent, like
    # cholesky_ex) and a finite-inputs flag are copied to pinned memory behind the factorisation and an event is
    # recorded.  The caller queues everything that follows (solves, inverse, sweep) and only then waits for that
    # event, so the GPU queue never drains; the jitter retry -- the rare path -- re-runs synchronously.
    def _launch_factorisation(self, ws, comps, scaled, noise, n):
        """Gram -> potrf of every latent in ws; info[:q] = first bad pivot, info[q] = non-finite-input flag.  Only
        queues device work, so graph 1 of the graphed step captures this same call."""
        q = noise.shape[0]
        K, dinv, info = ws["K"], ws["dinv"], ws["info"]
        # psd_safe_cholesky refuses a matrix with NaN entries before it factors anything.  Every entry of K is a
        # function of zn, Z, the outputscale and the noise, so the O(qn) inputs are checked instead of the n^2
        # matrix (the integer tensor path would turn a NaN into an arbitrary finite number, not propagate it).
        finite = torch.isfinite(noise).all()
        for c, (Z, zn, _, _) in zip(comps, scaled):
            finite = finite & torch.isfinite(zn).all()
            for t in (c[3], ops.shape_of(c)):
                if t is not None:
                    finite = finite & torch.isfinite(t).all()
        self.generation += 1
        self._gram_all(comps, scaled, noise, K, n)
        self._mark("gram")
        ops.potrf(K, dinv, info[:q], self.cfg_main)
        info[q:] = (~finite).to(torch.int32)

    def _status_copy(self, info):
        """Copies info into the engine's pinned buffer behind the queued work and records an event: (event, host
        view), the view valid once the event has completed."""
        if self._pinned is None or self._pinned.numel() != info.numel():
            self._pinned = torch.empty((info.numel(),), dtype=torch.int32).pin_memory()
        self._pinned.copy_(info, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return ev, self._pinned

    def _resolve_factorisation(self, status, ws, comps, scaled, noise, n, max_tries):
        """Wait for the factorisation's status (from _status_copy); returns True if a jitter retry re-factorised K
        (everything queued after the first attempt must then be redone)."""
        q = noise.shape[0]
        K, dinv, info = ws["K"], ws["dinv"], ws["info"]
        ev, host = status
        ev.synchronize()
        host = host.clone()
        if int(host[q]) != 0:
            raise NanError("cholesky: the kernel matrix contains NaN (non-finite inputs, lengthscales, outputscale "
                           "or noise)")
        bad = host[:q]
        if not bool(bad.any()):
            self.last_jitter = None
            return False

        def refactor(l, jitter):
            sl = slice(l, l + 1)
            da = (noise[sl] + jitter[sl]).contiguous()
            self.generation += 1
            self._gram_all(comps, scaled, da, K[sl], n, sl)
            ops.potrf(K[sl], dinv[sl], info[sl], self.cfg_main)

        # a failed member left garbage in its K; the others may have been overwritten by work queued after
        # the factorisation (the inverse runs in place), so every member is rebuilt, jitter only where needed
        self.last_jitter = self._jitter_retry(bad, info[:q], refactor, max_tries, rebuild_all_first=True)
        return True

    @staticmethod
    def _jitter_retry(bad, info, refactor, max_tries, rebuild_all_first):
        """psd_safe_cholesky's schedule after a failed batched factorisation (bad = host copy of info): jitter
        cholesky_jitter * 10^i on the members that still fail, a RuntimeWarning per retry, NotPSDError at the end.
        refactor(l, jitter) rebuilds member l with jitter[l] added to its diagonal and factorises it into info[l].
        Returns the jitter per member."""
        q = bad.shape[0]
        jitter = torch.zeros(q, dtype=torch.float64, device=info.device)
        base = settings.cholesky_jitter.value()
        prev_bad = bad
        new = 0.0
        first = rebuild_all_first
        for i in range(max_tries):
            new = base * (10**i)
            warnings.warn(f"A not p.d., added jitter of {new:.1e} to the diagonal", RuntimeWarning)
            members = range(q) if first else torch.nonzero(prev_bad).flatten().tolist()
            failing = set(torch.nonzero(prev_bad).flatten().tolist())
            for l in members:
                if l in failing:
                    jitter[l] = new
                refactor(l, jitter)
            first = False
            # members that were fine stay fine (same matrix); only previously failing ones can still fail
            prev_bad = info.cpu()
            if not bool(prev_bad.any()):
                return jitter
        raise NotPSDError(f"Matrix not positive definite after repeatedly adding jitter up to {new:.1e}.")

    # -- training: log-probabilities and all partial gradients -------------------
    def log_prob_and_grads(self, X, TY, comps, noise, need_grad, max_tries=None):
        """lp [q] = log N(TY_l; 0, sum_g o_gl k_gl(X,X) + noise_l I) for comps = [(kernel id, dims, ell [q, d_g],
        os [q] | None)] and, if need_grad, (dlp/dTY [q,n], dlp/dnoise [q], [dlp/dell_0, (dlp/dos_0), dlp/dell_1, ...])."""
        if max_tries is None:
            max_tries = settings.cholesky_max_tries.value()
        n, d = X.shape
        q = noise.shape[0]
        ws = self.workspace(X.device, q, n)
        np_ = ws["K"].shape[1]
        if need_grad and self.profile is None and 0 < np_ <= self.graph_max_order and X.is_cuda \
                and not self.capture_mode and not self._force_eager:
            key = (X.data_ptr(), X._version, tuple(X.shape), q,
                   tuple((c[0], tuple(c[1]), c[3] is not None, ops.shape_of(c) is not None) for c in comps),
                   self._cfg_key)
            if key in self._graphs:
                return self._log_prob_and_grads_graphed(ws, key, X, TY, comps, noise, max_tries)
            # the first call with these inputs, kernel structure and arithmetic runs eagerly (lazy library
            # initialisation must not happen under capture); the next one captures
            self._graphs[key] = "warm"
        self._mark("start")
        scaled = self._scaled(X, comps, np_)
        self._launch_factorisation(ws, comps, scaled, noise, n)
        if self.capture_mode:
            # the caller captures the whole training step into a CUDA graph (training.fit): no host wait in here;
            # it reads ws["info"] (first bad pivot per latent + the non-finite flag) after every replay and
            # repeats a failed iteration eagerly, where the jitter retry below applies
            self.capture_info = ws["info"]
            return self._solve_inverse_sweep(ws, comps, scaled, TY, n, need_grad)
        status = self._status_copy(ws["info"])
        self._mark("potrf")
        # queued behind the factorisation before its status is known
        out = self._solve_inverse_sweep(ws, comps, scaled, TY, n, need_grad)
        if self._resolve_factorisation(status, ws, comps, scaled, noise, n, max_tries):
            self._mark("retry")
            # a jitter retry re-factorised K: redo what depended on it
            out = self._solve_inverse_sweep(ws, comps, scaled, TY, n, need_grad)
        return out

    def _solve_inverse_sweep(self, ws, comps, scaled, TY, n, need_grad):
        """The step behind the factorisation in ws: (lp, None) or (lp, (dlp/dTY, dlp/dnoise, [dlp/dell_0, (dlp/dos_0),
        ...])).  Only queues device work, so graph 2 of the graphed step captures this same call."""
        # z, alpha, the quadratic form and the log-determinant come from L itself (two HBM-bound block
        # substitutions, csrc/trsv.cu) at full FP64-grade accuracy.  The explicit inverse K^-1 = L^-T L^-1
        # (trtri + lauum, 2/3 of the flops of the iteration) then feeds ONLY the gradient sweep
        # tr((alpha alpha^T - K^-1) dK), so both steps may run at the reduced cfg_kinv precision.
        K, dinv = ws["K"], ws["dinv"]
        z, alpha, quad, logdet = ops.solve_logdet(K, dinv, TY, n, ws["rhs"])
        lp = -0.5 * (quad + logdet + n * math.log(2 * math.pi))
        self._mark("solve_logdet")
        if not need_grad:
            return lp, None
        self.generation += 1
        ops.trtri(K, dinv, self.cfg_kinv)
        ops.lauum(K, dinv, self.cfg_kinv)
        self._mark("potri")
        g_noise, g_tensors = None, []
        for c, (Z, zn, _, _) in zip(comps, scaled):   # one sweep of K^-1 per additive component
            kid, dims, ell, os_ = c
            shape = ops.shape_of(c)
            g = ops.grad_sweep(K, alpha, Z, zn, ell, kid, os_, n, shape=shape)
            g_noise = g[2] if g_noise is None else g_noise
            g_tensors.append(g[0])
            if os_ is not None:
                g_tensors.append(g[1])
            if shape is not None:
                g_tensors.append(g[3])
        self._mark("grad_sweep")
        return lp, (-alpha, g_noise, g_tensors)

    @contextlib.contextmanager
    def _forced_eager(self):
        """Steps inside the block run on the eager path, never through the engine-level CUDA graphs."""
        was, self._force_eager = self._force_eager, True
        try:
            yield
        finally:
            self._force_eager = was

    # -- the same step as two replayed CUDA graphs (small problems) ---------------------------------------------
    def _log_prob_and_grads_graphed(self, ws, key, X, TY, comps, noise, max_tries):
        """Graph 1: scale -> Gram -> potrf.  Graph 2: solves -> inverse -> sweep(s).  Inputs are copied into static
        buffers, outputs cloned out of them; the status copy sits between the two replays, so the host waits for
        the factorisation only after the rest has been queued -- as in the eager path.  The call after the eager
        warm-up of `key` captures, later ones replay.  A failed factorisation falls back to the eager retry loop."""
        n = X.shape[0]
        st = self._graphs[key]
        if st == "warm":
            st = self._capture(ws, X, TY, comps, noise, n)
            self._graphs[key] = st
        # refresh the static inputs, replay
        st["TY"].copy_(TY)
        st["noise"].copy_(noise)
        for c, static in zip(comps, st["params"]):
            for src, dst in zip((c[2], c[3], ops.shape_of(c)), static):
                if src is not None:
                    dst.copy_(src)
        self.generation += 1
        st["g1"].replay()
        status = self._status_copy(ws["info"])
        self.generation += 1
        st["g2"].replay()
        ops.stats_add(st["launches"])            # the library kernels inside the two graphs
        lp, (neg_alpha, g_noise, g_tensors) = st["out"]
        out = (lp.clone(), (neg_alpha.clone(), g_noise.clone(), [g.clone() for g in g_tensors]))
        if self._resolve_factorisation(status, ws, st["comps"], st["scaled"], st["noise"], n, max_tries):
            # jitter retry re-factorised K eagerly: finish the step eagerly as well
            out = self._solve_inverse_sweep(ws, st["comps"], st["scaled"], TY, n, True)
        return out

    def _capture(self, ws, X, TY, comps, noise, n):
        TY_s, noise_s = TY.clone(), noise.clone()
        # static copies of (ell, os, shape parameter) of every component, refreshed before each replay
        params = [tuple(None if t is None else t.clone() for t in (c[2], c[3], ops.shape_of(c))) for c in comps]
        comps_s = [ops.Component(c[0], c[1], e, o, a) for c, (e, o, a) in zip(comps, params)]
        for kid, dims, _, _ in comps_s:
            self._sub_inputs(X, dims)            # column subsets / means are cached outside the graphs
        torch.cuda.synchronize(X.device)
        g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        launches0 = ops.stats_get()[0]
        with no_gc_during_capture(), torch.cuda.graph(g1):
            scaled = self._scaled(X, comps_s, ws["K"].shape[1])
            self._launch_factorisation(ws, comps_s, scaled, noise_s, n)
        with no_gc_during_capture(), torch.cuda.graph(g2, pool=g1.pool()):
            out = self._solve_inverse_sweep(ws, comps_s, scaled, TY_s, n, True)
        return dict(g1=g1, g2=g2, TY=TY_s, noise=noise_s, params=params, comps=comps_s, scaled=scaled, out=out,
                    launches=ops.stats_get()[0] - launches0)

    # -- optional phase timing (CUDA events on the launch stream; used by bench.py) --
    profile = None

    def _mark(self, name):
        if self.profile is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.profile.append((name, ev))

    def phase_ms(self):
        """Sum of the recorded phase durations (ms) by name; call after a synchronize."""
        out = {}
        prev = None
        for name, ev in self.profile or []:
            if name != "start" and prev is not None:
                out[name] = out.get(name, 0.0) + prev.elapsed_time(ev)
            prev = ev
        return out

    # -- dense noisy train covariance (kernel_cond, projected_lmc.py:367-369; small n only) --------
    def dense_gram(self, X, comps, noise):
        n, d = X.shape
        q = noise.shape[0]
        ws = self.workspace(X.device, q, n)
        np_ = ws["K"].shape[1]
        scaled = self._scaled(X, comps, np_)
        self.generation += 1
        self._gram_all(comps, scaled, noise, ws["K"], n)
        K = ws["K"][:, :n, :n]
        return torch.tril(K) + torch.tril(K, -1).transpose(1, 2)

    # -- leave-one-out by-product (projected_lmc.py:1108-1119) ----------------------
    def loo(self, X, TY, comps, noise, max_tries=None):
        n = X.shape[0]
        ws, _, alpha = self._factorise_and_solve(X, TY, comps, noise, max_tries)
        K, dinv = ws["K"], ws["dinv"]
        self.generation += 1
        ops.potri(K, dinv, self.cfg_main)
        sigma2 = 1.0 / torch.diagonal(K, dim1=1, dim2=2)[:, :n]
        return sigma2, alpha * sigma2

    def _factorise_and_solve(self, X, TY, comps, noise, max_tries):
        """Gram -> potrf with the jitter retry -> alpha = K^-1 TY, synchronously: (ws, scaled inputs, alpha)."""
        if max_tries is None:
            max_tries = settings.cholesky_max_tries.value()
        n = X.shape[0]
        ws = self.workspace(X.device, noise.shape[0], n)
        scaled = self._scaled(X, comps, ws["K"].shape[1])
        self._launch_factorisation(ws, comps, scaled, noise, n)
        status = self._status_copy(ws["info"])
        self._mark("potrf")
        self._resolve_factorisation(status, ws, comps, scaled, noise, n, max_tries)
        _, alpha, _, _ = ops.solve_logdet(ws["K"], ws["dinv"], TY, n, ws["rhs"])
        return ws, scaled, alpha

    # -- prediction -----------------------------------------------------------------
    def factorize(self, X, TY, comps, noise, max_tries=None):
        """Prediction cache: L (in ws['K']), dinv, alpha, scaled inputs of every kernel component."""
        n, d = X.shape
        q = noise.shape[0]
        ws, scaled, alpha = self._factorise_and_solve(X, TY, comps, noise, max_tries)
        prior_var = None                      # k(x*, x*) = sum_g os_g k_g(0) = sum_g os_g (1 without a ScaleKernel)
        for kid, dims, ell, os_ in comps:
            v = torch.ones(q, dtype=torch.float64, device=X.device) if os_ is None else os_
            prior_var = v if prior_var is None else prior_var + v
        return dict(L=ws["K"], dinv=ws["dinv"], alpha=alpha, comps=comps, scaled=scaled, prior_var=prior_var.contiguous(),
                    n=n, d=d, q=q, generation=self.generation)

    def state_is_current(self, st) -> bool:
        """False once anything (training step, compute_loo, kernel_cond, another factorize) has rewritten the
        shared workspace the prediction state points into."""
        return st is not None and st.get("generation") == self.generation and self._ws is not None and \
            st["L"].data_ptr() == self._ws["K"].data_ptr()

    def _check_state(self, st, device):
        """Refuses a stale prediction state and sets up the arithmetic for its order: (q, npad)."""
        if not self.state_is_current(st):
            raise RuntimeError("stale prediction state: the engine workspace was rewritten after factorize()")
        q, np_ = st["q"], st["L"].shape[1]
        self._configure_fp64(device, np_, q)
        return q, np_

    @staticmethod
    def tile_points(q: int, np_: int, budget_bytes: int = None, device=None) -> int:
        """Test points per cross-Gram tile [q, npad, mt]: as wide as the GEMMs like (8192) when a quarter of the
        free HBM holds the tile, never below what 6 GB hold."""
        if budget_bytes is None:
            budget_bytes = 6 << 30
            if device is not None and torch.cuda.is_available():
                budget_bytes = max(budget_bytes, torch.cuda.mem_get_info(device)[0] // 4)
        mt = (budget_bytes // (q * np_ * 8) // 128) * 128
        return int(max(128, min(8192, mt)))

    # Predictive variances need V = L^-1 K*.  A triangular SOLVE recurses down to 128-leaves (K = 128 products,
    # FP64-pipe bound); with the explicit inverse X = L^-1 (plmc_trtri_batched, n^3/3 per latent, once per
    # parameter state) V = X K* is a triangular MULTIPLY with dense 512-leaves: the same q n^2 n* FLOP at GEMM
    # speed.  "auto": invert once the points predicted with this state reach n/2 (the break-even of the extra
    # n^3/3); True / False force either path.
    predict_inverse = {"0": False, "1": True}.get(__import__("os").environ.get("PLMC_PREDICT_INVERSE", "auto"), "auto")

    def _maybe_invert(self, st, ns):
        if st.get("inverted"):
            return True
        st["points"] = st.get("points", 0) + ns
        want = self.predict_inverse
        if want == "auto":
            want = st["points"] * 2 >= st["n"]
        if want:
            ops.trtri(st["L"], st["dinv"], self.cfg_main)      # L -> L^-1 in place (alpha is already computed)
            st["inverted"] = True
        return bool(want)

    def predict_latents(self, st, Xs, need_var=True, tile=None):
        """Latent posterior means / variances at Xs: ([q, n*], [q, n*])."""
        q, np_ = self._check_state(st, Xs.device)
        ns = Xs.shape[0]
        dev = Xs.device
        mt_full = tile or self.tile_points(q, np_, device=dev)
        inverted = self._maybe_invert(st, ns) if need_var else False
        lat_mean = torch.empty((q, ns), dtype=torch.float64, device=dev)
        lat_var = torch.empty((q, ns), dtype=torch.float64, device=dev) if need_var else None
        Kx = None
        for s0 in range(0, ns, mt_full):
            cnt = min(mt_full, ns - s0)
            mt = _npad(cnt)
            if Kx is None or Kx.shape[2] != mt:
                Kx = None
                Kx = torch.empty((q, np_, mt), dtype=torch.float64, device=dev)
            lat_mean[:, s0:s0 + cnt] = self._cross_mean_v(st, Xs[s0:s0 + cnt], Kx, mt, inverted, need_var)[:, :cnt]
            if need_var:
                lat_var[:, s0:s0 + cnt] = ops.latent_var(Kx, st["prior_var"], mt)[:, :cnt]
        return lat_mean, lat_var

    def predict_latents_grad(self, st, Xs, g_mean=None, g_var=None, tile=None):
        """Gradient w.r.t. the test points Xs [n*, d] of sum_lj g_mean[l,j] mu_l(j) + g_var[l,j] v_l(j) for latent
        cotangents [q, n*] (either may be None): [n*, d].  Nothing is kept from the forward: each tile rebuilds K*
        and, with variance cotangents only, beta = K^-1 K* = L^-T (L^-1 K*) in place (trmm by the explicit inverse
        once the state is inverted, else trsm), so the memory is that of one prediction tile."""
        q, np_ = self._check_state(st, Xs.device)
        ns, d = Xs.shape
        dev = Xs.device
        out = torch.zeros((ns, d), dtype=torch.float64, device=dev)
        if g_mean is None and g_var is None:
            return out
        g_mean = None if g_mean is None else g_mean.contiguous()
        g_var = None if g_var is None else g_var.contiguous()
        mt_full = tile or self.tile_points(q, np_, device=dev)
        inverted = bool(st.get("inverted"))
        n = st["n"]
        Kx = None
        for s0 in range(0, ns, mt_full):
            cnt = min(mt_full, ns - s0)
            mt = _npad(cnt)
            if Kx is None or Kx.shape[2] != mt:
                Kx = None
                Kx = torch.empty((q, np_, mt), dtype=torch.float64, device=dev)
            xs = Xs[s0:s0 + cnt]
            scaled_t = []
            for g, (c, (_, _, _, xm)) in enumerate(zip(st["comps"], st["scaled"])):
                kid, dims, ell, os_ = c
                Zt, znt = ops.scale_inputs(self._component_inputs(xs, dims), xm, ell, mt)
                scaled_t.append((Zt, znt))
                if g_var is not None:
                    ops.cross_gram(st["scaled"][g][0], st["scaled"][g][1], Zt, znt, kid, os_, Kx, n, mt,
                                   accumulate=(g > 0), shape=ops.shape_of(c))
            beta = None
            if g_var is not None:
                if inverted:
                    ops.trmm(2, st["L"], st["dinv"], Kx, 1.0, self.cfg_main)
                    ops.trmm(3, st["L"], st["dinv"], Kx, 1.0, self.cfg_main)
                else:
                    ops.trsm(2, st["L"], st["dinv"], Kx, 1.0, self.cfg_main)
                    ops.trsm(3, st["L"], st["dinv"], Kx, 1.0, self.cfg_main)
                beta = Kx
            gm = None if g_mean is None else g_mean[:, s0:s0 + cnt]
            gv = None if g_var is None else g_var[:, s0:s0 + cnt]
            for c, (Z, zn, _, _), (Zt, znt) in zip(st["comps"], st["scaled"], scaled_t):
                kid, dims, ell, os_ = c
                gx = ops.cross_grad(Z, zn, Zt, znt, kid, os_, ell, st["alpha"], n, cnt, gm, gv, beta,
                                    shape=ops.shape_of(c))
                if tuple(dims) == tuple(range(d)):
                    out[s0:s0 + cnt] += gx
                else:
                    out[s0:s0 + cnt].index_add_(1, torch.as_tensor(list(dims), device=dev), gx)
        return out

    @staticmethod
    def _component_inputs(xs, dims):
        if len(dims) == xs.shape[1] and tuple(dims) == tuple(range(xs.shape[1])):
            return xs
        return xs.index_select(1, torch.as_tensor(list(dims), device=xs.device)).contiguous()

    def _cross_mean_v(self, st, xs, Kx, mt, inverted, need_v, zero_padding=False):
        """Cross-Gram K* of the test points xs into Kx [q, npad, mt], the latent means K*^T alpha [q, mt] (returned)
        and, if need_v, V = L^-1 K* in place (trmm by the explicit inverse once the state is inverted, else trsm).
        zero_padding: the columns of the padding test points are zeroed before the solve, so that V^T V has
        exact zeros outside the ns x ns block."""
        n = st["n"]
        for g, (c, (Z, zn, _, xm)) in enumerate(zip(st["comps"], st["scaled"])):
            kid, dims, ell, os_ = c
            Zt, znt = ops.scale_inputs(self._component_inputs(xs, dims), xm, ell, mt)
            ops.cross_gram(Z, zn, Zt, znt, kid, os_, Kx, n, mt, accumulate=(g > 0), shape=ops.shape_of(c))
        lat_mean = ops.latent_mean(Kx, st["alpha"], n, mt)
        if need_v:
            if zero_padding:
                Kx[:, :, xs.shape[0]:].zero_()
            if inverted:
                ops.trmm(2, st["L"], st["dinv"], Kx, 1.0, self.cfg_main)
            else:
                ops.trsm(2, st["L"], st["dinv"], Kx, 1.0, self.cfg_main)
        return lat_mean

    # -- joint posterior (full covariance, draws, joint log-density) -------------------------------------------
    # The n* test points are one tile; every buffer below belongs to the joint computation (the factor in ws["K"],
    # its dinv and the prediction state are only read).
    def latent_covariance(self, st, Xs):
        """Latent posterior means [q, n*] and covariances C = K** - V^T V as the lower 128-tiles of [q, m, m]
        (m = npad(n*), identity padding)."""
        q, np_ = self._check_state(st, Xs.device)
        ns = Xs.shape[0]
        dev = Xs.device
        m = _npad(ns)
        inverted = self._maybe_invert(st, ns)
        V = torch.empty((q, np_, m), dtype=torch.float64, device=dev)
        lat_mean = self._cross_mean_v(st, Xs, V, m, inverted, True, zero_padding=True)[:, :ns].contiguous()
        C = torch.empty((q, m, m), dtype=torch.float64, device=dev)
        zero = torch.zeros(q, dtype=torch.float64, device=dev)
        for g, (c, (_, _, _, xm)) in enumerate(zip(st["comps"], st["scaled"])):
            kid, dims, ell, os_ = c
            Zs, zns = ops.scale_inputs(self._component_inputs(Xs, dims), xm, ell, m)
            ops.gram(Zs, zns, kid, os_, zero, C, ns, accumulate=(g > 0), shape=ops.shape_of(c))
        ops.syrk(V, C, -1.0, 1.0, self.cfg_main)
        return lat_mean, C

    def factor_covariance(self, C, ns, max_tries=None):
        """Lower Cholesky factors of the latent covariances C [q, m, m] (a new tensor; C is kept), with
        psd_safe_cholesky's jitter schedule on the latents whose factorisation fails."""
        if max_tries is None:
            max_tries = settings.cholesky_max_tries.value()
        q, m, _ = C.shape
        Lc = C.clone()
        dinv = ops.alloc_dinv(m, q, C.device)
        info = torch.zeros(q, dtype=torch.int32, device=C.device)
        ops.potrf(Lc, dinv, info, self.cfg_main)
        bad = info.cpu()
        if bool(bad.any()):
            def refactor(l, jitter):
                Lc[l].copy_(C[l])
                Lc[l].diagonal()[:ns] += jitter[l]
                ops.potrf(Lc[l:l + 1], dinv[l:l + 1], info[l:l + 1], self.cfg_main)

            self._jitter_retry(bad, info, refactor, max_tries, rebuild_all_first=False)
        return Lc, dinv

    def latent_draws(self, Lc, dinv, normals):
        """chol(C_l) eps_l for normals [q, n*, S]: [q, m, npad(S)] (rows >= n* and columns >= S are padding)."""
        q, m, _ = Lc.shape
        _, ns, S = normals.shape
        G = torch.zeros((q, m, _npad(S)), dtype=torch.float64, device=Lc.device)
        G[:, :ns, :S] = normals
        ops.trmm(2, Lc, dinv, G, 1.0, self.cfg_main)
        return G

    def sample_latents(self, lat_mean, Lc, dinv, normals):
        """Latent posterior draws mean_l + chol(C_l) eps_l: [q, n*, S] for given normals [q, n*, S]."""
        ns, S = normals.shape[1], normals.shape[2]
        return self.latent_draws(Lc, dinv, normals)[:, :ns, :S] + lat_mean[:, :, None]

    def joint_log_prob(self, C, H, S, mean, values, max_tries=None):
        """log N(values; mean, sum_l C_l (x) h_l h_l^T + I (x) S) for values [B, n*, p] (mean [n*, p]): [B]."""
        B, ns, p = values.shape
        N = ns * p
        T = ops.task_covariance(C, H, S, ns, tiled=True)
        L, dinv = self.factor_covariance(T, N, max_tries)
        del T                                 # only the factor is used from here on
        resid = (values - mean).reshape(B, N)
        if B == 1:
            z, _, quad, logdet = ops.solve_logdet(L, dinv, resid.contiguous(), N)
        else:
            Z = torch.zeros((1, L.shape[1], _npad(B)), dtype=torch.float64, device=L.device)
            Z[0, :N, :B] = resid.T
            ops.trsm(2, L, dinv, Z, 1.0, self.cfg_main)
            quad = Z[0, :N, :B].pow(2).sum(0)
            logdet = 2.0 * L[0].diagonal()[:N].log().sum()
        return -0.5 * (quad + logdet + N * math.log(2 * math.pi))
