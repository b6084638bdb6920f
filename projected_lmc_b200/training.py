"""Training-loop helper: the loop of the reference drivers (experiments.py:259-284,
realdata_experiments.py:174-210) around the CUDA path -- AdamW, exponential learning-rate decay,
plateau-based early stop -- without the per-iteration host synchronisation.

The reference calls ``loss.item()`` every iteration to evaluate its stopping rule
(experiments.py:275); here losses stay on the device and the same rule is evaluated over a
buffered history every ``check_every`` iterations.  Inside an iteration the only host wait is on
the event recorded right after the Cholesky factorisation (its per-latent status decides on the
psd_safe_cholesky jitter retry); it is taken AFTER the solves, the inverse and the gradient
sweep of the same iteration have been queued behind it, so the GPU queue does not drain on it
(engine.LatentEngine.log_prob_and_grads).

Launch-bound problems (BASELINE config 1: n = 1000, 50 tasks, 10 latents -- ~3.7 ms of kernels behind ~5.5 ms of host
work per iteration) run the WHOLE iteration as two replayed CUDA graphs (``cuda_graph``): graph 1 = forward +
backward (mixing-matrix QR, projection, Gram, Cholesky, solves, inverse, sweep, projection terms and their autograd),
graph 2 = AdamW step + learning-rate decay.  Between the two the host reads the factorisation status of that
iteration; a failed factorisation is repeated eagerly with gpytorch's jitter-retry semantics before graph 2 runs.
"""
from __future__ import annotations

import time
import warnings
from typing import Optional

import numpy as np
import torch

from . import gp, ops
from .engine import no_gc_during_capture


def _invalidate_data_caches(eng, mll):
    """Forget everything derived from the contents of X and Y (column means, per-component input subsets, S = Y^T Y)."""
    eng._forget_inputs()
    if hasattr(mll, "_S_key"):
        mll._S_key = None


class _GraphedStep:
    """One training iteration as two CUDA graphs (see the module docstring).  Built after a few eager iterations
    (lazy library initialisation, optimiser state and every host-side cache must exist before capture)."""

    def __init__(self, model, mll, X, Y, optimizer, lr_t, gamma, hist, max_tries):
        self.model, self.mll, self.X, self.Y, self.opt = model, mll, X, Y, optimizer
        self.eng = model._engine
        self.hist, self.max_tries = hist, max_tries
        self.params = [p for p in model.parameters() if p.requires_grad]
        dev = X.device
        self.it_t = torch.zeros(1, dtype=torch.long, device=dev)
        torch.cuda.synchronize(dev)
        self.g1, self.g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        optimizer.zero_grad(set_to_none=True)
        # everything derived from X and Y (column means, per-component input subsets, S = Y^T Y) is recomputed INSIDE
        # the graph, so a caller may refresh the contents of X / Y in place between replays
        _invalidate_data_caches(self.eng, mll)
        # nothing may keep the autograd graph of an earlier (eager) iteration alive: its AccumulateGrad nodes belong
        # to the stream they were created on, and synchronising with that stream is not allowed during capture
        if getattr(mll, "proj_term_list", None) is not None:
            mll.proj_term_list = None
        self.eng.capture_mode = True
        launches0 = ops.stats_get()[0]
        try:
            with no_gc_during_capture(), torch.cuda.graph(self.g1):
                loss = -mll(model(X), Y)
                loss.backward()
                hist.index_copy_(0, self.it_t, loss.detach().reshape(1).to(hist.dtype))
                self.it_t.add_(1)
            self.loss = loss.detach()
            self.info = self.eng.capture_info
            with no_gc_during_capture(), torch.cuda.graph(self.g2, pool=self.g1.pool()):
                optimizer.step()
                if lr_t is not None and gamma is not None:
                    lr_t.mul_(gamma)          # ExponentialLR, chained form: lr <- lr * gamma
        finally:
            self.eng.capture_mode = False
        self.launches = ops.stats_get()[0] - launches0      # library kernels inside graph 1 (per replay)
        if self.info is None:
            raise RuntimeError("the model's latent term did not run on the engine during capture")

    def set_iteration(self, it):
        self.it_t.fill_(it)

    def run(self, it):
        """Iteration `it`: returns nothing; the loss is written to hist[it] on the device."""
        self.eng.capture_mode = True          # (replays launch nothing from Python; the flag guards re-entrancy)
        try:
            self.g1.replay()
        finally:
            self.eng.capture_mode = False
        self.eng.generation += 2              # the replay rewrote the engine workspace (prediction caches)
        ops.stats_add(self.launches)
        ev, host = self.eng._status_copy(self.info)
        ev.synchronize()
        if int(host[-1]) != 0 or bool(host[:-1].any()):
            # failed factorisation (or non-finite inputs): repeat this iteration on the eager path, which applies
            # psd_safe_cholesky's jitter schedule (or raises NanError / NotPSDError); gradients go into the SAME
            # static .grad buffers graph 2 reads
            for p in self.params:
                if p.grad is not None:
                    p.grad.zero_()
            with self.eng._forced_eager():
                loss = -self.mll(self.model(self.X), self.Y)
                loss.backward()
            self.hist[it] = loss.detach()
        self.g2.replay()


def fit(model, mll, X, Y, n_iter: int, lr: float = 1e-2, lr_min: Optional[float] = 1e-3, loss_thresh: float = 1e-4,
        patience: int = 500, check_every: int = 25, cholesky_max_tries: int = 8, optimizer=None, scheduler=None,
        print_loss: bool = False, freq_print: int = 100, sync_grads=None, cuda_graph="auto", graph_warmup: int = 3):
    """Train ``model`` by maximising ``mll``; returns a dict with the loss history and timings.

    Stopping rule of the reference: ``|1 - loss_i / loss_{i-1}| < loss_thresh`` for more than
    ``patience`` consecutive iterations.  ``sync_grads(loss, params)`` is called after backward in
    latent-parallel runs (``distributed.allreduce_loss_and_grads``)."""
    # whole-step CUDA graphs: only with the optimiser / schedule built here (AdamW must be `capturable`, the decay must
    # live on the device), a single process, the exact (non-inducing) model and a matrix order the engine calls small
    eng = getattr(model, "_engine", None)
    want_graph = cuda_graph is True or cuda_graph == "auto"
    can_graph = (want_graph and X.is_cuda and optimizer is None and scheduler is None and sync_grads is None
                 and eng is not None and getattr(model, "_inducing", lambda: None)() is None
                 and (cuda_graph is True or 0 < ((X.shape[0] + 127) // 128) * 128 <= eng.graph_max_order)
                 and n_iter > graph_warmup + 1)
    lr_t, gamma = None, None
    if lr_min is not None:
        gamma = float(np.exp(np.log(lr_min / lr) / n_iter))
    if optimizer is None:
        if can_graph:
            lr_t = torch.tensor(float(lr), dtype=torch.float64, device=X.device)
            optimizer = torch.optim.AdamW(model.parameters(), lr=lr_t, capturable=True)
        else:
            optimizer = torch.optim.AdamW(model.parameters(), lr=lr)
    if scheduler is None and lr_min is not None and not can_graph:
        scheduler = torch.optim.lr_scheduler.ExponentialLR(optimizer, gamma=gamma)
    params = [p for p in model.parameters() if p.requires_grad]
    model.train()
    losses = torch.empty(n_iter, dtype=torch.float64, device=X.device)
    plateau_id, last, checked, stop_at = 0, None, 0, None
    start = time.time()
    it = 0
    graphed, graph_note = None, None
    if can_graph and X is not model.train_inputs[0]:
        # model(X) compares X with the training inputs unless it IS that tensor -- a device comparison with a host
        # read, which cannot be captured: compare once here and pass the model's own tensor from then on
        tx = model.train_inputs[0]
        if X.shape == tx.shape and X.dtype == tx.dtype and (X.data_ptr() == tx.data_ptr() or torch.equal(X, tx)):
            X = tx
        else:
            can_graph = False                  # (the model will refuse these inputs on the first iteration)
    with gp.settings.cholesky_max_tries(cholesky_max_tries):
        for it in range(n_iter):
            if can_graph and graphed is None and it == graph_warmup:
                loss = None                    # drop the last eager iteration's autograd graph before capturing
                try:
                    graphed = _GraphedStep(model, mll, X, Y, optimizer, lr_t, gamma, losses, cholesky_max_tries)
                except Exception as ex:  # noqa: BLE001  (an op of this torch build that cannot be captured)
                    torch.cuda.synchronize(X.device)
                    can_graph, graph_note = False, repr(ex)[:200]
                    # what the aborted capture cached was recorded, never computed
                    _invalidate_data_caches(eng, mll)
                    warnings.warn("the training step could not be captured into a CUDA graph; continuing with eager "
                                  f"launches ({graph_note})", RuntimeWarning)
                    try:
                        # a capture that ended in an error leaves torch's CUDA generator flagged as capturing (every
                        # later random draw would fail); a trivial successful capture clears the flag
                        with torch.cuda.graph(torch.cuda.CUDAGraph()):
                            torch.zeros(1, device=X.device)
                    except Exception:  # noqa: BLE001
                        pass
            if graphed is not None:
                graphed.set_iteration(it) if it == graph_warmup else None
                graphed.run(it)
            else:
                optimizer.zero_grad(set_to_none=True)
                loss = -mll(model(X), Y)
                loss.backward()
                if sync_grads is not None:
                    loss = sync_grads(loss, params)
                optimizer.step()
                if scheduler is not None:
                    scheduler.step()
                elif lr_t is not None and gamma is not None:
                    lr_t.mul_(gamma)           # device-resident ExponentialLR (eager warm-up / fallback iterations)
                losses[it] = loss.detach()
            if (it + 1) % check_every == 0 or it == n_iter - 1:
                hist = losses[checked:it + 1].tolist()        # one host sync per check_every iterations
                for k, new in enumerate(hist, start=checked):
                    if print_loss and k % freq_print == 0:
                        print(new)
                    if k > 0 and abs(1 - new / last) < loss_thresh:
                        plateau_id += 1
                        if plateau_id > patience and stop_at is None:
                            stop_at = k
                    else:
                        plateau_id = 0
                    last = new
                checked = it + 1
                if stop_at is not None:
                    break
    if X.is_cuda:
        torch.cuda.synchronize()
    n_done = it + 1
    return {"losses": losses[:n_done].cpu(), "n_iter": n_done, "stopped_at": stop_at,
            "train_time": time.time() - start, "cuda_graph": graphed is not None, "cuda_graph_note": graph_note}
