"""Batched box-constrained LTI MPC on the GPU (``lqr_b200.mpc``).

``BoxMPC(A, B, Q, R, rho)`` builds the ADMM cache of ``lqrb_admm_cache_f64`` once (the DARE of the rho-augmented costs
and the factor every iteration reuses) and keeps it, with the ADMM state, on the device.  ``.solve(x0, ...)`` runs
``lqrb_admm_solve_f64``: per instance, with x_1 = x0,

    min  sum_{k<N} 1/2 |x_k - xref_k|_Q^2 + 1/2 |u_k - uref_k|_R^2 + 1/2 |x_N - xref_N|_Qf^2
    s.t. x_{k+1} = A x_k + B u_k,  umin_k <= u_k <= umax_k (k = 1..N-1),  xmin_k <= x_k <= xmax_k (k = 2..N)

THE TERMINAL COST DEPENDS ON rho: Qf = Pt - rho I with Pt = DARE(A, B, Q + rho I, R + rho I) (``self.Qf``); it is what
lets one cached factor serve every iteration.  The returned trajectory is the last ADMM iterate: dynamically exact and
within the primal residual of the bounds.

Shapes (CUDA float64 tensors, batch first, math order; a batch of 1 is broadcast):
    A (b, n, n)  B (b, n, m)  Q (b, n, n)  R (b, m, m)   (Q and R are read through their upper triangles)
    x0 (b, n)  xref (b, N, n)  uref (b, N-1, m)  umin / umax (b, N-1, m)  xmin / xmax (b, N-1, n) (knots 2..N)
    ->  X (b, N, n), U (b, N-1, m), info (b,) int32: 0 converged, 1 max_iter reached, 2 NaN input or iterate (X, U NaN),
        3 an empty box (X, U NaN).
Every argument after x0 may be None (reference 0, bound +-inf) or anything that broadcasts to its shape (a float, a
(m,) vector, ...).  N is taken from the per-knot arguments, or given as ``N=`` when there are none.  ``warm=True``
starts from the ADMM state the previous call left (same N and batch): the receding-horizon loop, where consecutive
problems differ little.  The state is not shifted by a knot between calls.  ``iters`` and ``res`` (r_pri, r_dual) of
the last call are kept as ``.iters``, ``.res``.  The calls run on the current torch stream and do not synchronise.

Not differentiable: no gradient flows through ``solve`` (the natural extension, implicit differentiation at the
active set, is not built).  There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import torch

from . import _lib, ops
from .autograd import _cm, _handle

__all__ = ["BoxMPC"]


def _check(t, what):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64):
        raise TypeError(f"BoxMPC takes CUDA float64 tensors ({what}); there is no CPU path")


class BoxMPC:
    def __init__(self, A, B, Q, R, rho: float):
        for k, t in zip("ABQR", (A, B, Q, R)):
            _check(t, k)
        self.device = A.device
        self.b = max(t.shape[0] for t in (A, B, Q, R))
        self.n, self.m = A.shape[-1], B.shape[-1]
        self.rho = float(rho)
        full = lambda t: _cm(t.expand((self.b,) + tuple(t.shape[1:])))  # noqa: E731
        self.cache = torch.empty(self.b, ops.admm_cache_doubles(self.n, self.m), dtype=torch.float64,
                                 device=self.device)
        self.cache_info = torch.empty(self.b, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            ops.admm_cache(_handle(self.device), self.n, self.m, self.b, self.rho, full(A), full(B), full(Q), full(R),
                           self.cache, self.cache_info)
        parts = ops.admm_cache_split(self.cache, self.n, self.m)
        self.K, self.Qf = parts["K"], parts["Qf"]
        self.state = None
        self.iters = self.res = None

    def solve(self, x0, xref=None, uref=None, umin=None, umax=None, xmin=None, xmax=None, max_iter: int = 100,
              eps: float = 1e-6, warm: bool = True, N: int | None = None):
        """One MPC solve; see the module docstring.  Returns (X, U, info)."""
        _check(x0, "x0")
        if self.b == 1 and x0.shape[0] > 1:  # one system for a batch of initial states: copy its record per instance
            self.b = x0.shape[0]
            self.cache = self.cache.expand(self.b, -1).contiguous()
            self.state = None
        n, m, b, dev = self.n, self.m, self.b, self.device
        knots = [t.shape[-2] + 1 for t in (uref, umin, umax, xmin, xmax) if isinstance(t, torch.Tensor) and t.dim() >= 2]
        if isinstance(xref, torch.Tensor) and xref.dim() >= 2:
            knots.append(xref.shape[-2])
        if N is None:
            if not knots:
                raise ValueError("N is needed when no per-knot argument gives it")
            N = knots[0]
        if any(k != N for k in knots):
            raise ValueError(f"per-knot arguments disagree on N: {knots} (N = {N})")

        def arg(t, rows, cols):
            if t is None:
                return None
            if isinstance(t, torch.Tensor):
                _check(t, "per-knot argument")
            t = torch.as_tensor(t, dtype=torch.float64, device=dev)
            return t.expand(b, rows, cols).contiguous()
        L = 2 * (N - 1) * (m + n)
        warm = warm and self.state is not None and self.state.shape == (b, L)
        if not warm:
            self.state = torch.empty(b, L, dtype=torch.float64, device=dev)
        Z = torch.empty(b, _lib.num_vars(n, m, N), dtype=torch.float64, device=dev)
        self.iters = torch.empty(b, dtype=torch.int32, device=dev)
        self.res = torch.empty(b, 2, dtype=torch.float64, device=dev)
        info = torch.empty(b, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            ops.admm_solve(_handle(dev), n, m, N, b, self.cache, x0.expand(b, n).contiguous(), Z, arg(xref, N, n),
                           arg(uref, N - 1, m), arg(umin, N - 1, m), arg(umax, N - 1, m), arg(xmin, N - 1, n),
                           arg(xmax, N - 1, n), self.state, warm, max_iter, eps, eps, self.iters, self.res, info)
        body = Z[:, :(N - 1) * (n + m)].view(b, N - 1, n + m)
        X = torch.cat([body[:, :, :n], Z[:, None, (N - 1) * (n + m):]], dim=1)
        return X, body[:, :, n:].contiguous(), info
