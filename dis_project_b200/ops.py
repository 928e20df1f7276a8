"""Device-level operators: torch CUDA tensors in, torch CUDA tensors out, CUDA kernels through the
C-ABI in between.  torch is plumbing only (device memory, streams); no torch op is on the compute
path.  All calls are stream-ordered on torch's current stream and do not synchronise.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, Optional, Tuple

import torch

from . import _lib

F64 = torch.float64


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev(t) -> torch.Tensor:
    """Accept numpy / torch input, return a contiguous fp64 CUDA tensor."""
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(t, dtype=F64)
    if t.dtype != F64:
        t = t.to(F64)
    if not t.is_cuda:
        _lib.require_device()
        t = t.cuda()
    return t.contiguous()


def _rows3(X: torch.Tensor, name: str) -> torch.Tensor:
    X = _dev(X)
    if X.ndim != 2 or X.shape[1] != 3:
        raise ValueError(f"{name} must have shape (n, 3) = [time, gene_index, flag] (dataset.py:391), got {tuple(X.shape)}")
    return X


def _check_training_flags(X) -> None:
    """The training covariance Sigma is built from k_xx only (every training row of the reference has flag 1,
    dataset.py:388; objectives.py:70 would blend the other branches in for flag-0 rows).  A host copy of X is checked
    here; a device-resident X is the caller's responsibility (include/lfm_b200.h, lfm_nlml)."""
    if isinstance(X, torch.Tensor):
        if X.is_cuda or X.ndim != 2 or X.shape[1] != 3:
            return
        bad = bool((X[:, 2] != 1).any())
    else:
        import numpy as np

        Xh = np.asarray(X)
        if Xh.ndim != 2 or Xh.shape[1] != 3:
            return
        bad = bool((Xh[:, 2] != 1).any())
    if bad:
        raise ValueError("training inputs must all carry flag 1 (gene expression rows): the objective and the "
                         "posteriors build Sigma from k_xx only")


def _theta(theta: torch.Tensor, G: int) -> torch.Tensor:
    theta = _dev(theta).reshape(-1)
    if theta.numel() != 3 * G + 2:
        raise ValueError(f"theta must hold 3G+2={3 * G + 2} values [d,s,b,l,sigma], got {theta.numel()}")
    return theta


_WS: Dict[Tuple[int, str], torch.Tensor] = {}


def _workspace(nbytes: int, device: torch.device, tag: str) -> torch.Tensor:
    key = (device.index if device.index is not None else torch.cuda.current_device(), tag)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        _WS.pop(key, None)
        buf = None
        buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


def release_workspaces() -> None:
    _WS.clear()


# ------------------------------------------------------------------------------------------------
def cross_covariance(X, Y, theta, G: int) -> torch.Tensor:
    """ExactLFM.cross_covariance(kernel, x, y) (reference src/model.py:372-394)."""
    X, Y = _rows3(X, "x"), _rows3(Y, "y")
    theta = _theta(theta, G)
    N, M = X.shape[0], Y.shape[0]
    out = torch.empty((N, M), dtype=F64, device=X.device)
    if N == 0 or M == 0:
        return out
    _lib.check(_lib.lib().lfm_cross_covariance(_stream(), N, M, X.data_ptr(), Y.data_ptr(), G, theta.data_ptr(),
                                               out.data_ptr(), M), "lfm_cross_covariance")
    return out


def gram(X, theta, G: int) -> torch.Tensor:
    """ExactLFM.gram(kernel, x) as a dense array (reference src/model.py:396-414)."""
    return cross_covariance(X, X, theta, G)


def h_terms(j, k, t1, t2, theta, G: int) -> torch.Tensor:
    """ExactLFM.h(j, k, t1, t2), elementwise (reference src/model.py:315-365)."""
    j, k, t1, t2 = (_dev(torch.as_tensor(a, dtype=F64).reshape(-1)) for a in (j, k, t1, t2))
    theta = _theta(theta, G)
    n = j.numel()
    out = torch.empty(n, dtype=F64, device=j.device)
    _lib.check(_lib.lib().lfm_h(_stream(), n, j.data_ptr(), k.data_ptr(), t1.data_ptr(), t2.data_ptr(), G,
                                theta.data_ptr(), out.data_ptr()), "lfm_h")
    return out


def mean_function(X, theta, G: int) -> torch.Tensor:
    """ExactLFM.mean_function(x) (reference src/model.py:124-149); shape (N, 1)."""
    X = _rows3(X, "x")
    theta = _theta(theta, G)
    N = X.shape[0]
    if N % G:
        raise ValueError(f"mean_function: {N} rows is not divisible by num_genes={G} (model.py:145-149)")
    out = torch.empty((N, 1), dtype=F64, device=X.device)
    _lib.check(_lib.lib().lfm_mean_function(_stream(), N, X.data_ptr(), G, theta.data_ptr(), out.data_ptr()),
               "lfm_mean_function")
    return out


def constrain(theta_unc, G: int) -> torch.Tensor:
    u = _dev(theta_unc)
    P = 3 * G + 2
    B = u.numel() // P
    out = torch.empty_like(u)
    _lib.check(_lib.lib().lfm_constrain(_stream(), B, G, u.data_ptr(), out.data_ptr()), "lfm_constrain")
    return out


def unconstrain(theta, G: int) -> torch.Tensor:
    t = _dev(theta)
    P = 3 * G + 2
    B = t.numel() // P
    out = torch.empty_like(t)
    _lib.check(_lib.lib().lfm_unconstrain(_stream(), B, G, t.data_ptr(), out.data_ptr()), "lfm_unconstrain")
    return out


_TG_CACHE: Dict[Tuple[int, int, int], int] = {}


def distinct_times(X) -> int:
    """Number of distinct times among the rows of X: the `time_grid` bound of the *_tg entry points.
    Counted on a host copy; for a device tensor the answer is remembered per (storage, version, rows), so a
    fit loop pays one device->host copy per data set, not per evaluation."""
    import numpy as np

    if isinstance(X, torch.Tensor):
        if X.is_cuda:
            key = (X.data_ptr(), X._version, X.shape[0])
            if key not in _TG_CACHE:
                if len(_TG_CACHE) > 64:
                    _TG_CACHE.clear()
                Xh = np.ascontiguousarray(X.detach().cpu().numpy(), dtype=np.float64)
                _TG_CACHE[key] = int(_lib.lib().lfm_count_distinct_times(Xh.shape[0], Xh.ctypes.data))
            return _TG_CACHE[key]
        Xh = X.detach().numpy()
    else:
        Xh = np.asarray(X)
    Xh = np.ascontiguousarray(Xh, dtype=np.float64)
    if Xh.ndim != 2 or Xh.shape[1] != 3:
        return 0
    return int(_lib.lib().lfm_count_distinct_times(Xh.shape[0], Xh.ctypes.data))


def _variances(variances, N: int) -> Optional[torch.Tensor]:
    if variances is None:
        return None
    v = _dev(variances).reshape(-1)
    if v.numel() != N:
        raise ValueError(f"variances has {v.numel()} values for {N} input rows")
    return v


def _nlml_call(fn_name: str, X, y, theta, jitter: float, G: int, nout: int, time_grid: Optional[int] = None,
               variances=None):
    if time_grid is None:
        time_grid = distinct_times(X)
    _check_training_flags(X)
    X = _rows3(X, "x")
    y = _dev(y).reshape(-1)
    theta = _theta(theta, G)
    N = X.shape[0]
    if y.numel() != N:
        raise ValueError(f"y has {y.numel()} values for {N} input rows")
    if N % G:
        raise ValueError(f"{N} rows is not divisible by num_genes={G} (model.py:145-149)")
    l = _lib.lib()
    nbytes = l.lfm_nlml_workspace_bytes_tg(N, G, int(time_grid))
    ws = _workspace(nbytes, X.device, "nlml")
    out = torch.empty(nout, dtype=F64, device=X.device)
    info = torch.zeros(1, dtype=torch.int32, device=X.device)
    v = _variances(variances, N)
    _lib.check(getattr(l, fn_name)(_stream(), N, G, X.data_ptr(), y.data_ptr(), v.data_ptr() if v is not None else None,
                                   theta.data_ptr(), float(jitter), int(time_grid), ws.data_ptr(), ws.numel(),
                                   out.data_ptr(), info.data_ptr()),
               fn_name)
    return out, info


class NlmlGradPlan:
    """One NLML+grad evaluation over fixed device buffers, captured once as a CUDA graph and replayed per call
    (include/lfm_b200.h, "evaluation plans").  What a fit loop wants: (X, y) stay, theta changes.

        plan = NlmlGradPlan(X, y, G, jitter)          # or unconstrained=True for trainer.py:126 semantics
        out, info = plan(theta)                        # out[0] = NLML, out[1:] = gradient; buffers are reused

    `out` / `info` are the plan's own buffers: copy them if they must survive the next call."""

    def __init__(self, X, y, G: int, jitter: float, unconstrained: bool = False, time_grid: Optional[int] = None,
                 variances=None):
        import ctypes as C

        if time_grid is None:
            time_grid = distinct_times(X)
        _check_training_flags(X)
        self.X = _rows3(X, "x")
        self.y = _dev(y).reshape(-1)
        self.G, self.P = int(G), 3 * int(G) + 2
        N = self.X.shape[0]
        if self.y.numel() != N:
            raise ValueError(f"y has {self.y.numel()} values for {N} input rows")
        if N % G:
            raise ValueError(f"{N} rows is not divisible by num_genes={G} (model.py:145-149)")
        self.variances = _variances(variances, N)   # heteroscedastic objective (include/lfm_b200.h)
        dev = self.X.device
        l = _lib.lib()
        self.theta = torch.ones(self.P, dtype=F64, device=dev)  # a valid point for the warm-up evaluation
        if not unconstrained:
            self.theta[3 * G] = 2.5
        self.out = torch.empty(self.P + 1, dtype=F64, device=dev)
        self.info = torch.zeros(1, dtype=torch.int32, device=dev)
        self.ws = torch.empty(int(l.lfm_nlml_workspace_bytes_tg(N, G, int(time_grid))), dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        self._plan = C.c_void_p()
        _lib.check(l.lfm_nlml_grad_plan_create_het(C.byref(self._plan), N, G, self.X.data_ptr(), self.y.data_ptr(),
                                                   self.variances.data_ptr() if self.variances is not None else None,
                                                   self.theta.data_ptr(), float(jitter), int(time_grid),
                                                   int(bool(unconstrained)), self.ws.data_ptr(), self.ws.numel(),
                                                   self.out.data_ptr(), self.info.data_ptr()),
                   "lfm_nlml_grad_plan_create_het")

    def __call__(self, theta):
        t = theta if isinstance(theta, torch.Tensor) else torch.as_tensor(theta, dtype=F64)
        if t.numel() != self.P:
            raise ValueError(f"theta must hold 3G+2={self.P} values [d,s,b,l,sigma], got {t.numel()}")
        self.theta.copy_(t.reshape(-1), non_blocking=True)
        _lib.check(_lib.lib().lfm_plan_launch(self._plan, _stream()), "lfm_plan_launch")
        return self.out, self.info

    def close(self) -> None:
        if getattr(self, "_plan", None):
            _lib.lib().lfm_plan_destroy(self._plan)
            self._plan = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


def nlml(X, y, theta, jitter: float, G: int, time_grid: Optional[int] = None, variances=None):
    """CustomConjMLL(negative=True) (reference src/objectives.py:21-78): (out[1] = NLML, info[1]).
    `variances` (N,) adds diag(variances) to Sigma: the heteroscedastic objective of the reference's GPyTorch twin
    (src/gpytorch_alfi/model_alfi.py:294-299)."""
    return _nlml_call("lfm_nlml_het_tg", X, y, theta, jitter, G, 1, time_grid, variances)


def nlml_grad(X, y, theta, jitter: float, G: int, time_grid: Optional[int] = None, variances=None):
    """NLML and its gradient w.r.t. the constrained theta: out[0] = NLML, out[1:] = gradient."""
    return _nlml_call("lfm_nlml_grad_het_tg", X, y, theta, jitter, G, 3 * G + 3, time_grid, variances)


def nlml_grad_unc(X, y, theta_unc, jitter: float, G: int, time_grid: Optional[int] = None, variances=None):
    """jax.value_and_grad(JaxTrainer.loss) w.r.t. the unconstrained leaves (reference src/trainer.py:126)."""
    return _nlml_call("lfm_nlml_grad_unc_het_tg", X, y, theta_unc, jitter, G, 3 * G + 3, time_grid, variances)


def latent_posterior(X, y, variances, theta, jitter: float, Xstar, G: int):
    """ExactLFM.latent_predict (reference src/model.py:420-463): returns (mean[T*], var[T*], info[1])."""
    _check_training_flags(X)
    X = _rows3(X, "x")
    Xs = _rows3(Xstar, "test_inputs")
    y = _dev(y).reshape(-1)
    variances = _dev(variances).reshape(-1)
    theta = _theta(theta, G)
    N, T = X.shape[0], Xs.shape[0]
    if y.numel() != N or variances.numel() != N:
        raise ValueError("y / variances do not match the number of training rows")
    if N % G:
        raise ValueError(f"{N} rows is not divisible by num_genes={G} (model.py:145-149)")
    l = _lib.lib()
    mean = torch.empty(T, dtype=F64, device=X.device)
    var = torch.empty(T, dtype=F64, device=X.device)
    info = torch.zeros(1, dtype=torch.int32, device=X.device)
    if T == 0:
        return mean, var, info
    nbytes = l.lfm_latent_posterior_workspace_bytes(N, G, T)
    ws = _workspace(nbytes, X.device, "post")
    _lib.check(l.lfm_latent_posterior(_stream(), N, G, X.data_ptr(), y.data_ptr(), variances.data_ptr(),
                                      theta.data_ptr(), float(jitter), T, Xs.data_ptr(), ws.data_ptr(), ws.numel(),
                                      mean.data_ptr(), var.data_ptr(), info.data_ptr()), "lfm_latent_posterior")
    return mean, var, info


def gene_posterior(X, y, variances, theta, jitter: float, Xstar, G: int, full_cov: bool = True):
    """ExactLFM.multi_gene_predict (reference src/model.py:465-514): (mean[T*], cov[T*,T*] or None, var[T*], info)."""
    _check_training_flags(X)
    X = _rows3(X, "x")
    Xs = _rows3(Xstar, "test_inputs")
    y = _dev(y).reshape(-1)
    variances = _dev(variances).reshape(-1)
    theta = _theta(theta, G)
    N, T = X.shape[0], Xs.shape[0]
    if y.numel() != N or variances.numel() != N:
        raise ValueError("y / variances do not match the number of training rows")
    if N % G or T % G:
        raise ValueError("mean_function: rows must be divisible by num_genes (model.py:145-149)")
    l = _lib.lib()
    mean = torch.empty(T, dtype=F64, device=X.device)
    var = torch.empty(T, dtype=F64, device=X.device)
    cov = torch.empty((T, T), dtype=F64, device=X.device) if full_cov else None
    info = torch.zeros(1, dtype=torch.int32, device=X.device)
    ws = _workspace(l.lfm_gene_posterior_workspace_bytes(N, G, T), X.device, "gene")
    _lib.check(l.lfm_gene_posterior(_stream(), N, G, X.data_ptr(), y.data_ptr(), variances.data_ptr(), theta.data_ptr(),
                                    float(jitter), T, Xs.data_ptr(), ws.data_ptr(), ws.numel(), mean.data_ptr(),
                                    cov.data_ptr() if full_cov else None, var.data_ptr(), info.data_ptr()),
               "lfm_gene_posterior")
    return mean, cov, var, info


def unique_rows(X) -> int:
    """Number of distinct (time, gene, flag) rows (host-side; X is at most 128 x 3 on this path)."""
    import numpy as np

    Xh = X.detach().cpu().numpy() if isinstance(X, torch.Tensor) else np.asarray(X, dtype=np.float64)
    Xh = np.ascontiguousarray(Xh, dtype=np.float64)
    return int(_lib.lib().lfm_count_unique_rows(Xh.shape[0], Xh.ctypes.data))


def _y_layout(shape, B: int, N: int) -> bool:
    """Shape of the observations of B batched LFMs: (B, N) -> True, one row per LFM; N values -> False, shared by every
    LFM.  Anything else raises ValueError."""
    shape = tuple(int(n) for n in shape)
    if shape == (B, N) and not (B == N == 1):
        return True
    if math.prod(shape) == N:
        return False
    raise ValueError(f"y must hold N={N} observations (shared) or be (B, N)=({B}, {N}) (one row per LFM), got {shape}")


def _batched_y(y, B: int, N: int) -> Tuple[torch.Tensor, int]:
    """y (N,) shared by every LFM -> (y, 0); y (B, N), one row of observations per LFM -> (y, N)."""
    y = _dev(y)
    return (y, N) if _y_layout(y.shape, B, N) else (y.reshape(-1), 0)


def _variance_layout(shape, B: int, N: int) -> bool:
    """Shape of the measurement variances of the batched heteroscedastic objective: (B, N) -> True, one row per LFM
    (mirrors `_batched_y`); (N,) or (N, 1) -> False, shared by every LFM.  Anything else raises ValueError."""
    shape = tuple(int(n) for n in shape)
    if shape == (B, N) and B != 1:
        return True
    if shape in ((N,), (N, 1)) or (B == 1 and shape == (1, N)):
        return False
    raise ValueError(f"variances must be (N,), (N, 1) with N={N} (shared) or (B, N)=({B}, {N}) (one row per LFM), "
                     f"got {shape}")


def _batched_variances(variances, B: int, N: int) -> Tuple[torch.Tensor, int]:
    """variances -> (device tensor, var_stride): 0 when shared, N when one row per LFM."""
    v = _dev(variances)
    return (v, N) if _variance_layout(v.shape, B, N) else (v.reshape(-1), 0)


def batched_nlml_grad_unc(X, y, theta_unc, jitter: float, G: int, time_grid: Optional[int] = None, variances=None):
    """B independent value_and_grad evaluations.  theta_unc (B, P) -> (val[B], grad[B,P], info[B]).
    y is (N,) -- every LFM sees the same observations -- or (B, N): LFM b sees y[b] (replicas / candidate TFs).
    `time_grid`: bound on the distinct times of X (None: counted from X; 0: one CTA per LFM, no tables).
    `variances`: None, or the measurement variances of the heteroscedastic objective (Sigma += diag(variances),
    include/lfm_b200.h, lfm_batched_nlml_grad_unc_het): (N,) / (N, 1) shared, or (B, N) one row per LFM."""
    hint = unique_rows(X)
    tg = distinct_times(X) if time_grid is None else int(time_grid)
    _check_training_flags(X)
    X = _rows3(X, "x")
    u = _dev(theta_unc)
    P = 3 * G + 2
    if u.ndim != 2 or u.shape[1] != P:
        raise ValueError(f"theta_unc must be (B, {P})")
    B, N = u.shape[0], X.shape[0]
    y, y_stride = _batched_y(y, B, N)
    v, v_stride = _batched_variances(variances, B, N) if variances is not None else (None, 0)
    val = torch.empty(B, dtype=F64, device=X.device)
    grad = torch.empty((B, P), dtype=F64, device=X.device)
    info = torch.zeros(B, dtype=torch.int32, device=X.device)
    if B == 0:
        return val, grad, info
    if v is not None:
        _lib.check(_lib.lib().lfm_batched_nlml_grad_unc_het(_stream(), B, N, G, X.data_ptr(), y.data_ptr(), y_stride,
                                                            v.data_ptr(), v_stride, u.data_ptr(), float(jitter), hint, tg,
                                                            val.data_ptr(), grad.data_ptr(), info.data_ptr()),
                   "lfm_batched_nlml_grad_unc_het")
        return val, grad, info
    _lib.check(_lib.lib().lfm_batched_nlml_grad_unc_multi(_stream(), B, N, G, X.data_ptr(), y.data_ptr(), y_stride,
                                                          u.data_ptr(), float(jitter), hint, tg, val.data_ptr(),
                                                          grad.data_ptr(), info.data_ptr()),
               "lfm_batched_nlml_grad_unc_multi")
    return val, grad, info


def _batched_posterior(fn_name: str, gene: bool, X, y, variances, theta, jitter: float, Xstar, G: int,
                       full_cov: bool):
    """Shared body of batched_latent_posterior / batched_gene_posterior (lfm_batched_*_posterior, include/lfm_b200.h)."""
    import numpy as np

    if variances is None:
        raise ValueError("variances are required (the posteriors' training covariance is K + diag(variances) + ...)")
    _check_training_flags(X)
    shape = lambda a: tuple(a.shape) if hasattr(a, "shape") else np.shape(a)   # checked before any device copy
    P = 3 * G + 2
    for name, s in (("x", shape(X)), ("test_inputs", shape(Xstar))):
        if len(s) != 2 or s[1] != 3:
            raise ValueError(f"{name} must have shape (n, 3) = [time, gene_index, flag] (dataset.py:391), got {s}")
    if len(shape(theta)) != 2 or shape(theta)[1] != P:
        raise ValueError(f"theta must be (B, {P}) constrained [d,s,b,l,sigma] rows, got {shape(theta)}")
    B, N, T = shape(theta)[0], shape(X)[0], shape(Xstar)[0]
    if shape(y) != (B, N) and int(np.prod(shape(y))) != N:
        raise ValueError(f"y must hold N={N} observations (shared) or be (B, N)=({B}, {N}) (one row per LFM), "
                         f"got {shape(y)}")
    _variance_layout(shape(variances), B, N)
    if N % G or (gene and T % G):
        raise ValueError("mean_function: rows must be divisible by num_genes (model.py:145-149)")
    hint = unique_rows(X)
    X, Xs, th = _rows3(X, "x"), _rows3(Xstar, "test_inputs"), _dev(theta)
    y, y_stride = _batched_y(y, B, N)
    v, v_stride = _batched_variances(variances, B, N)
    dev = X.device
    mean = torch.empty((B, T), dtype=F64, device=dev)
    var = torch.empty((B, T), dtype=F64, device=dev)
    cov = torch.empty((B, T, T), dtype=F64, device=dev) if full_cov else None
    info = torch.zeros(B, dtype=torch.int32, device=dev)
    if B == 0 or (T == 0 and not gene):
        return mean, cov, var, info
    l = _lib.lib()
    ws = _workspace(max(int(l.lfm_batched_posterior_workspace_bytes(B, N, G, T, hint, int(bool(full_cov)))), 16), dev,
                    "bpost")
    args = [_stream(), B, N, G, X.data_ptr(), y.data_ptr(), y_stride, v.data_ptr(), v_stride, th.data_ptr(),
            float(jitter), T, Xs.data_ptr(), hint, ws.data_ptr(), ws.numel(), mean.data_ptr()]
    if gene:
        args.append(cov.data_ptr() if full_cov else None)
    args += [var.data_ptr(), info.data_ptr()]
    _lib.check(getattr(l, fn_name)(*args), fn_name)
    return mean, cov, var, info


def batched_latent_posterior(X, y, variances, theta, jitter: float, Xstar, G: int):
    """ExactLFM.latent_predict (reference src/model.py:420-463) of B LFMs in one launch: theta (B, P) constrained (e.g.
    MultiStartResult.theta), y (N,) or (B, N), variances (N,), (N, 1) or (B, N).  Returns (mean (B, T*), var (B, T*),
    info (B,)); info as lfm_batched_latent_posterior (include/lfm_b200.h), a failed LFM has NaN outputs."""
    mean, _, var, info = _batched_posterior("lfm_batched_latent_posterior", False, X, y, variances, theta, jitter, Xstar,
                                            G, False)
    return mean, var, info


def batched_gene_posterior(X, y, variances, theta, jitter: float, Xstar, G: int, full_cov: bool = False):
    """ExactLFM.multi_gene_predict (reference src/model.py:465-514) of B LFMs in one launch; arguments as
    batched_latent_posterior.  Returns (mean (B, T*), cov (B, T*, T*) or None, var (B, T*), info (B,))."""
    return _batched_posterior("lfm_batched_gene_posterior", True, X, y, variances, theta, jitter, Xstar, G,
                              bool(full_cov))


class BatchedFitState:
    """Device-resident state of B independent fits (iterates, Adam moments, loss history).

    ONE device allocation [u | adam | theta | hist | info | extra] and ONE initialisation launch
    (lfm_batched_fit_init); `n_keys` int64 words at the start of `extra` are set to INT64_MAX (best-objective keys)."""

    def __init__(self, theta0, G: int, total_steps: int, extra_doubles: int = 0, n_keys: int = 0, keys_offset: int = 0,
                 B: Optional[int] = None, device=None):
        """`theta0` None with `B` and `device`: allocate only (a cached state that `reset` re-initialises per fit)."""
        self.G, self.P = G, 3 * G + 2
        if theta0 is not None:
            theta0 = _dev(theta0)
            if theta0.ndim != 2 or theta0.shape[1] != self.P:
                raise ValueError(f"theta0 must be (B, {self.P}) constrained start points")
            B, device = theta0.shape[0], theta0.device
        self.B = int(B)
        self.total_steps = int(total_steps)
        dev = device
        # everything a caller reads back lives behind the iterate and the moments (theta | hist | info | extra), so that
        # the results of a fit cross PCIe as one copy (batched_to_host)
        S = max(1, self.total_steps)
        n_u = self.B * self.P
        n_theta, n_hist, n_info = n_u, self.B * S, (self.B + 1) // 2
        self._cuts = (n_theta, n_theta + n_hist, n_theta + n_hist + n_info)
        whole = torch.empty(3 * n_u + self._cuts[2] + int(extra_doubles), dtype=F64, device=dev)
        self.u = whole[:n_u].view(self.B, self.P)
        self.adam = whole[n_u:3 * n_u].view(self.B, 2 * self.P)
        self.blob = whole[3 * n_u:]
        self.theta = self.blob[:n_theta].view(self.B, self.P)
        self.hist = self.blob[n_theta:self._cuts[1]].view(self.B, S)
        self.info = self.blob[self._cuts[1]:self._cuts[2]].view(torch.int32)[:self.B]
        self.extra = self.blob[self._cuts[2]:]
        if n_keys > int(extra_doubles) - int(keys_offset):
            raise ValueError("the best-objective keys live inside `extra`")
        keys = self.extra[keys_offset:keys_offset + n_keys].view(torch.int64) if n_keys else None
        # arguments of lfm_batched_fit_init behind (stream, B, G, theta0)
        self._init_tail = (self.u.data_ptr(), self.adam.data_ptr(), self.hist.data_ptr(), n_hist, self.info.data_ptr(),
                           keys.data_ptr() if n_keys else None, n_keys)
        self.unique_hint = 0  # filled from X on the first batched_fit_steps call
        self.time_grid = None  # distinct-time bound, counted from X on the first call (0: CTA-per-LFM kernel)
        self.struct_cache = None  # device bytes that carry the structure of X from the first launch to the later ones
        self.queue_ws = None      # task queue of the persistent mode (batched_fit_steps(queue_chunk=...))
        self.step = 0
        if theta0 is not None:
            self.reset(theta0)

    def reset(self, theta0: torch.Tensor) -> None:
        """(Re-)initialise the state for a fit from the constrained start points `theta0` (B x P, device): ONE launch."""
        self.step = 0
        if self.B:
            _lib.check(_lib.lib().lfm_batched_fit_init(_stream(), self.B, self.G, theta0.data_ptr(), *self._init_tail),
                       "lfm_batched_fit_init")


_PINNED: Dict[int, torch.Tensor] = {}


def _pinned(n: int) -> torch.Tensor:
    buf = _PINNED.get(n)
    if buf is None:
        buf = torch.empty(n, dtype=F64, pin_memory=True)
        _PINNED[n] = buf
    return buf


def batched_to_host(state: "BatchedFitState", after_copy=None):
    """(theta, hist, info, extra) of a fit as numpy arrays: ONE device->host copy through a cached pinned buffer.
    `after_copy`: a torch.cuda.Event recorded right behind the copy (device-side timing of a whole fit)."""
    host = _pinned(state.blob.numel())
    host.copy_(state.blob, non_blocking=True)
    if after_copy is not None:
        after_copy.record()
    torch.cuda.current_stream().synchronize()
    a = host.numpy()
    c0, c1, c2 = state._cuts
    theta = a[:c0].reshape(state.B, state.P).copy()
    hist = a[c0:c1].reshape(state.B, -1).copy()
    info = a[c1:c2].view("int32")[:state.B].copy()
    return theta, hist, info, a[c2:].copy()


def batched_best(hist: Optional[torch.Tensor], col: int, theta: Optional[torch.Tensor], id0: float,
                 out: torch.Tensor) -> None:
    """out (P + 2) = [loss, id0 + b, theta_b] of the restart b with the smallest finite hist[b, col] (one launch)."""
    P = out.numel() - 2
    B = 0 if hist is None else hist.shape[0]
    _lib.check(_lib.lib().lfm_batched_best(_stream(), B, P, hist.data_ptr() if B else None,
                                           hist.stride(0) if B else max(col + 1, 1), int(col),
                                           theta.data_ptr() if B else None, float(id0), out.data_ptr()),
               "lfm_batched_best")


def loss_key_to_float(keys):
    """Inverse of the order-preserving double -> int64 map of include/lfm_b200.h (best_key); INT64_MAX -> inf."""
    import numpy as np

    k = np.asarray(keys, dtype=np.int64)
    bits = np.where(k >= 0, k, k ^ np.int64(0x7FFFFFFFFFFFFFFF))
    out = bits.view(np.float64).copy()
    out[k == np.iinfo(np.int64).max] = np.inf
    return out


def _structure_cache(state: BatchedFitState, N: int, device) -> None:
    """The device bytes that carry the structure of X from the first launch of a fit to the later ones, sized for the
    state's unique-row hint and distinct-time bound (grown, never shrunk)."""
    nb = max(int(_lib.lib().lfm_batched_structure_bytes(N, state.G, state.unique_hint, int(state.time_grid))), 16)
    if state.struct_cache is None or state.struct_cache.numel() < nb:
        state.struct_cache = torch.empty(nb, dtype=torch.uint8, device=device)


def _bind_fit(state: BatchedFitState, X: torch.Tensor, y: torch.Tensor, y_stride: int, v: Optional[torch.Tensor],
              var_stride: int, jitter: float, lr: float, b1: float, b2: float, eps: float, fix_params: bool,
              steps_per_epoch: int, step_keys: Optional[torch.Tensor], queue_chunk: int):
    """lfm_batched_fit_het over `state` with every argument bound but the stream, the step range and `best_key`: returns
    launch(stream, first_step, steps, best_key_ptr).  Bound once per fit, so that a launch per optimiser step costs one
    ctypes call.  `queue_chunk` > 0 only when one launch runs the whole fit: persistent workers over a device-side queue
    of `queue_chunk`-step tasks (include/lfm_b200.h; the library ignores the queue where it does not pay)."""
    l = _lib.lib()
    qb = int(l.lfm_batched_queue_bytes(state.B, state.total_steps, int(queue_chunk))) if queue_chunk > 0 else 0
    if qb > 0 and (state.queue_ws is None or state.queue_ws.numel() < qb):
        state.queue_ws = torch.empty(qb, dtype=torch.uint8, device=X.device)
    head = (state.B, X.shape[0], state.G, X.data_ptr(), y.data_ptr(), y_stride, v.data_ptr() if v is not None else None,
            var_stride, state.u.data_ptr(), state.adam.data_ptr(), float(jitter), float(lr), float(b1), float(b2),
            float(eps))
    mid = (state.total_steps, int(bool(fix_params)), int(steps_per_epoch), state.unique_hint, int(state.time_grid),
           state.hist.data_ptr(), state.hist.shape[1], state.theta.data_ptr(), state.info.data_ptr())
    tail = (step_keys.data_ptr() if step_keys is not None else None, state.struct_cache.data_ptr(),
            int(queue_chunk) if qb > 0 else 0, state.queue_ws.data_ptr() if qb > 0 else None, qb)
    fit, check = l.lfm_batched_fit_het, _lib.check

    def launch(stream: int, first_step: int, steps: int, best_key: Optional[int]) -> None:
        check(fit(stream, *head, first_step, steps, *mid, best_key, *tail), "lfm_batched_fit_het")

    return launch


def batched_fit_steps(state: BatchedFitState, X, y, jitter: float, steps: int, *, lr: float = 0.01,
                      b1: float = 0.9, b2: float = 0.999, eps: float = 1e-8, fix_params: bool = True,
                      steps_per_epoch: int = 1000, best_key: Optional[torch.Tensor] = None,
                      step_keys: Optional[torch.Tensor] = None, queue_chunk: int = 0, variances=None) -> None:
    """Advance every fit in `state` by `steps` optimiser steps (reference src/trainer.py:201-216).
    y is (N,) (multi-start: one data set, B start points) or (B, N) (one row of observations per LFM).
    `variances`: None, or the measurement variances of the heteroscedastic objective, (N,) / (N, 1) shared or (B, N)
    one row per LFM (lfm_batched_fit_het, include/lfm_b200.h).
    `best_key`: one int64 device word, atomicMin of the loss keys after the last step of this call; `step_keys`:
    total_steps int64 device words, word s = atomicMin of the loss keys at step s (include/lfm_b200.h).
    `queue_chunk` > 0 with the whole fit in this one call: persistent workers over a task queue of `queue_chunk`-step
    tasks (the queue mode of lfm_batched_fit_het)."""
    if state.unique_hint == 0:
        state.unique_hint = unique_rows(X)
        _check_training_flags(X)
    if state.time_grid is None:
        state.time_grid = distinct_times(X)
    X = _rows3(X, "x")
    y, y_stride = _batched_y(y, state.B, X.shape[0])
    v, v_stride = _batched_variances(variances, state.B, X.shape[0]) if variances is not None else (None, 0)
    if state.B == 0 or steps <= 0:
        return
    steps = min(steps, state.total_steps - state.step)
    _structure_cache(state, X.shape[0], X.device)
    if step_keys is not None and step_keys.numel() < state.total_steps:
        raise ValueError("step_keys must hold one int64 word per step of the fit")
    whole = state.step == 0 and steps == state.total_steps
    launch = _bind_fit(state, X, y, y_stride, v, v_stride, jitter, lr, b1, b2, eps, fix_params, steps_per_epoch,
                       step_keys, queue_chunk if whole else 0)
    launch(_stream(), state.step, steps, best_key.data_ptr() if best_key is not None else None)
    state.step += steps


def debug_dgemm_nt(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """C = A B^T through the library's DMMA kernel (roofline helper)."""
    A, B = _dev(A), _dev(B)
    M, K = A.shape
    N = B.shape[0]
    Cm = torch.empty((M, N), dtype=F64, device=A.device)
    _lib.check(_lib.lib().lfm_debug_dgemm_nt(_stream(), M, N, K, A.data_ptr(), B.data_ptr(), Cm.data_ptr()),
               "lfm_debug_dgemm_nt")
    return Cm


GEMM_KMODES = {"full": 0, "le_row": 1, "ge_row": 3, "ge_rowcol": 4, "lauum_late": 5}


def debug_dgemm(A: torch.Tensor, B: torch.Tensor, C: torch.Tensor, M: int, N: int, K: int, *, lda: int, ldb: int,
                ldc: int, transA: int = 0, transB: int = 0, offA: int = 0, offB: int = 0, offC: int = 0,
                alpha: float = 1.0, beta: float = 0.0, lower_only: bool = False, kmode: int = 0, batch: int = 1,
                strideA: int = 0, strideB: int = 0, strideC: int = 0, tile: int = 0, tri_skip: int = 0,
                k_split: int = 0, k_lo: int = 0, k_hi: int = 1 << 62) -> int:
    """One launch of the dense path's DMMA GEMM (lfm_debug_dgemm, include/lfm_b200.h) over 1-D float64 CUDA buffers.
    Operands start at element offsets offA / offB / offC of their buffers; pass the same buffer and offset for C and A
    to multiply in place.  Returns the code of the instantiation that ran (TA TBN WM WN GM as decimal digits); a
    descriptor the library refuses raises _lib.LfmError with its status.  Raises ValueError, before calling the
    library, if any element an operand could be read or written at lies outside its buffer."""
    nb = batch if batch > 1 else 1
    ops_ = (("A", A, offA, lda, strideA, (K, M) if transA else (M, K)),
            ("B", B, offB, ldb, strideB, (N, K) if transB else (K, N)),
            ("C", C, offC, ldc, strideC, (M, N)))
    for name, buf, off, ld, stride, (rows, cols) in ops_:
        if not (isinstance(buf, torch.Tensor) and buf.is_cuda and buf.dtype == F64 and buf.ndim == 1
                and buf.is_contiguous()):
            raise ValueError(f"{name} must be a contiguous 1-D float64 CUDA tensor")
        if min(off, ld, stride) < 0:
            raise ValueError(f"{name}: negative offset, leading dimension or stride")
        if rows > 0 and cols > 0 and off + (nb - 1) * stride + (rows - 1) * ld + cols - 1 >= buf.numel():
            raise ValueError(f"{name}: a {rows} x {cols} operand (ld {ld}, {nb} problems, stride {stride}) at offset "
                             f"{off} reaches past the buffer's {buf.numel()} elements")
    d = _lib.GemmDesc(transA=int(transA), transB=int(transB), M=M, N=N, K=K,
                      A=A.data_ptr() + 8 * offA, lda=lda, B=B.data_ptr() + 8 * offB, ldb=ldb,
                      C=C.data_ptr() + 8 * offC, ldc=ldc, alpha=alpha, beta=beta, lower_only=int(lower_only),
                      kmode=kmode, batch=batch, strideA=strideA, strideB=strideB, strideC=strideC, tile=tile,
                      tri_skip=tri_skip, k_split=k_split, k_lo=k_lo, k_hi=k_hi)
    variant = ctypes.c_int(0)
    _lib.check(_lib.lib().lfm_debug_dgemm(_stream(), ctypes.byref(d), ctypes.byref(variant)), "lfm_debug_dgemm")
    return variant.value


def _scratch_like(A: torch.Tensor, W: Optional[torch.Tensor]) -> torch.Tensor:
    if W is None:
        return torch.zeros_like(A)
    if not (W.is_cuda and W.dtype == F64 and W.shape == A.shape and W.is_contiguous()):
        raise ValueError(f"W must be a contiguous float64 CUDA tensor of shape {tuple(A.shape)}")
    return W


def debug_potrf_potri(A: torch.Tensor, want_inverse: bool = True, W: Optional[torch.Tensor] = None):
    """In-place Cholesky (+ inverse) of a dense SPD matrix; returns (L, Sinv_lower or None, info).  `W` (n x n, may be
    None) is the scratch the library works in: after the call its lower triangle holds W = L^-1 when want_inverse."""
    A = _dev(A)
    n = A.shape[0]
    W = _scratch_like(A, W)
    Sinv = torch.zeros_like(A) if want_inverse else None
    info = torch.zeros(1, dtype=torch.int32, device=A.device)
    _lib.check(_lib.lib().lfm_debug_potrf_potri(_stream(), n, A.data_ptr(), W.data_ptr(),
                                                Sinv.data_ptr() if want_inverse else None, info.data_ptr()),
               "lfm_debug_potrf_potri")
    return A, Sinv, info


def debug_factor_inverse_eval(A: torch.Tensor, chain_ready: bool = True, W: Optional[torch.Tensor] = None):
    """The factorisation and Sigma^-1 in the sequence the NLML gradient runs them (lfm_debug_potrf_potri_eval), in place:
    returns (Sinv_lower (= A), W = L^-1 (lower), diag(L), early_done, info)."""
    A = _dev(A)
    n = A.shape[0]
    W = _scratch_like(A, W)
    ldiag = torch.empty(n, dtype=F64, device=A.device)
    info = torch.zeros(1, dtype=torch.int32, device=A.device)
    early = ctypes.c_int(0)
    _lib.check(_lib.lib().lfm_debug_potrf_potri_eval(_stream(), n, A.data_ptr(), W.data_ptr(), ldiag.data_ptr(),
                                                     int(bool(chain_ready)), ctypes.byref(early), info.data_ptr()),
               "lfm_debug_potrf_potri_eval")
    return A, W, ldiag, bool(early.value), info
