"""``JaxTrainer``: the optimiser loop of the reference (``src/trainer.py:36-228``).

Same constructor and ``fit`` signature.  Each step is one fused NLML+gradient evaluation on the
B200 (``CustomConjMLL.value_and_grad``) followed by the optax-style update on the 3G+2 leaves; the
"fix p21" hook fires exactly where the reference's does (after the update of every step with
``step % num_steps_per_epoch == 0`` in UNCONSTRAINED space, and once more in constrained space after
the loop; SURVEY.md Q5).  When the problem is small enough for the batched kernel (N <= 128) and the
optimiser is ``adam``, the whole scan runs inside a single persistent CUDA kernel.
"""
from __future__ import annotations

from typing import Any, Optional

import numpy as np

from . import ops
from .gpx_compat import Dataset, GradientTransformation, apply_updates
from .model import ExactLFM
from .objectives import CustomConjMLL


class JaxTrainer:
    def __init__(self, model: ExactLFM, objective, training_data: Dataset, optim: GradientTransformation,
                 key: Any, num_iters: int, track_parameters: Optional[list] = None):
        self.model = model.unconstrain()  # reference trainer.py:75
        self.objective = objective
        self.training_data = training_data
        self.optim = optim
        self.key = key
        self.num_iters = int(num_iters)
        self.track_parameters = {k: [] for k in track_parameters} if track_parameters else None
        self.history = []

    def loss(self, model: ExactLFM, batch: Dataset) -> float:
        """objective(model.constrain(), batch) for an unconstrained model (reference trainer.py:86-103)."""
        model = model.stop_gradient()
        return self.objective(model.constrain(), batch)

    def step(self, carry: tuple, key: Any, step_count: int) -> tuple:
        """One optimiser step (reference trainer.py:105-131): value_and_grad, update, apply."""
        model, opt_state = carry
        batch = self.training_data
        if hasattr(self.objective, "value_and_grad"):
            loss_val, loss_gradient = self.objective.value_and_grad(model, batch)
        else:
            raise NotImplementedError("the objective must provide value_and_grad (no tracing autodiff here)")
        updates, opt_state = self.optim.update(loss_gradient, opt_state, model)
        model = apply_updates(model, updates)
        return (model, opt_state), loss_val

    def after_epoch_jax(self, model: ExactLFM, fix_params: Optional[bool]) -> ExactLFM:
        """Pin sensitivity[3] = 1 and decay[3] = 0.8 (p21) in whatever space `model` is in
        (reference trainer.py:133-160).  Out-of-range index 3 is dropped, as JAX's .at[].set does."""
        if not fix_params or model.num_genes <= 3:
            return model
        s = np.array(model.true_s, dtype=np.float64)
        d = np.array(model.true_d, dtype=np.float64)
        s[3] = 1.0
        d[3] = 0.8
        return model.replace(true_s=s, true_d=d)

    def _device_scan_ok(self) -> bool:
        n = self.training_data.n
        return (isinstance(self.objective, CustomConjMLL) and self.objective.negative
                and isinstance(self.optim, GradientTransformation) and self.optim.name == "adam"
                # with variances the fit stays the host loop of dense evaluations (the batched kernels have the
                # heteroscedastic objective too, lfm_batched_fit_het, but this path is not routed to them)
                and getattr(self.objective, "variances", None) is None
                and n <= 128 and n % self.model.num_genes == 0 and not self.track_parameters)

    def fit(self, fix_params: Optional[bool] = True, num_steps_per_epoch: Optional[int] = 1000) -> tuple:
        """Run `num_iters` steps; returns (constrained model, loss history) like the reference
        (``trainer.fit``, reference trainer.py:162-228)."""
        if self._device_scan_ok():
            # the whole lax.scan as one persistent kernel (B = 1 restart)
            theta0 = self.model.constrain().pack()[None, :]
            st = ops.BatchedFitState(theta0, self.model.num_genes, self.num_iters)
            ops.batched_fit_steps(st, self.training_data.X, np.asarray(_host(self.training_data.y)).reshape(-1),
                                  self.model.jitter, self.num_iters, lr=self.optim.learning_rate, b1=self.optim.b1,
                                  b2=self.optim.b2, eps=self.optim.eps, fix_params=bool(fix_params),
                                  steps_per_epoch=int(num_steps_per_epoch))
            theta, hist, info, _ = ops.batched_to_host(st)
            if int(info[0]) < 0:  # the kernel refused the problem (not a numerical failure, which gives NaN like JAX)
                raise RuntimeError(f"batched fit kernel refused the problem (info = {int(info[0])})")
            self.model = self.model.with_leaves(theta[0])
            self.history = hist[0]
        else:
            state = self.optim.init(self.model)
            model = self.model
            history = np.empty(self.num_iters)
            for step_count in range(self.num_iters):
                (model, state), loss_val = self.step((model, state), None, step_count)
                if step_count % num_steps_per_epoch == 0:
                    model = self.after_epoch_jax(model, fix_params)
                history[step_count] = loss_val
            model = model.constrain()
            self.model = self.after_epoch_jax(model, fix_params) if fix_params else model
            self.history = history
        if self.track_parameters:
            return self.model, self.history, self.track_parameters
        return self.model, self.history


def _host(a):
    try:
        import torch

        if isinstance(a, torch.Tensor):
            return a.detach().cpu().numpy()
    except Exception:  # pragma: no cover
        pass
    return a
