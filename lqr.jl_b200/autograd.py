"""Differentiable batched Riccati solve for torch (``lqr_b200.autograd``).

``riccati_solve(A, B, Q, R, q, r, Qf, qf, x0, N=None) -> (X, U, info)`` solves the LTV-affine LQR of
``lqrb_riccati_f64`` on CUDA float64 tensors in math order and backpropagates through it with
``lqrb_riccati_grad_f64``: the adjoint of an LQR is another LQR with the same matrices, so the backward pass is one
more solve on the same kernels plus one sweep that forms the gradients.

Shapes (math order, batch first):
    LTV:  A (b, N-1, n, n)  B (b, N-1, n, m)  Q (b, N-1, n, n)  R (b, N-1, m, m)  q (b, N-1, n)  r (b, N-1, m)
    LTI:  A (b, n, n)       B (b, n, m)       Q (b, n, n)       R (b, m, m)       q (b, n)       r (b, m)   and N given
    Qf (b, n, n)  qf (b, n)  x0 (b, n)          ->  X (b, N, n), U (b, N-1, m), info (b,) int32
An argument with batch size 1 is broadcast over the batch (autograd sums its gradient).  q, r, qf may be None
(zero).  Q, R and Qf are symmetrised first (the solve reads their upper triangles), so the gradients are exact for
non-symmetric inputs too.  ``info`` is the potrf info of the solve (0 = ok) and is not differentiable; the gradients
of an instance with info != 0 carry no meaning.  The calls run on the current torch stream and do not synchronise;
calls on different streams are ordered one after another (they share the device's handle).
There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from . import _lib, ops

__all__ = ["riccati_solve"]


def _cm(a):
    """math order (..., rows, cols) -> contiguous column-major buffer"""
    return a.transpose(-1, -2).contiguous()


_CUDA_STREAM_LEGACY = 1  # cudaStreamLegacy: torch's default stream, which the ABI's NULL (the handle's own) is not

# One handle per device, owned by this module (ops.default_handle keeps its own stream).  A handle's scratch serves
# every call made on it, whatever the stream, so a call issued on another torch stream than the handle's previous
# call is first ordered after that stream; otherwise it could repack the scratch that call is still reading.
_handles: dict[int, list] = {}  # device index -> [Handle, torch stream of its last call]


def _handle(device: torch.device) -> _lib.Handle:
    st = _handles.get(device.index)
    if st is None:
        st = _handles[device.index] = [_lib.Handle(device.index), None]
    h, last = st
    cur = torch.cuda.current_stream(device)
    if last is not None and last != cur:
        cur.wait_stream(last)
    st[1] = cur
    h.set_stream(cur.cuda_stream or _CUDA_STREAM_LEGACY)
    return h


class _RiccatiSolve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, N, A, B, Q, R, q, r, Qf, qf, x0):
        b, n, m = x0.shape[0], A.shape[-1], B.shape[-1]
        flags = _lib.FLAG_LTI if A.dim() == 3 else 0
        args = [_cm(A), _cm(B), _cm(Q), _cm(R), q, r, _cm(Qf), qf]
        Z = torch.empty(b, _lib.num_vars(n, m, N), dtype=torch.float64, device=x0.device)
        info = torch.empty(b, dtype=torch.int32, device=x0.device)
        with torch.cuda.device(x0.device):
            ops.riccati(_handle(x0.device), n, m, N, b, flags, *args, x0, Z, None, None, info)
        ctx.save_for_backward(*[a if a is not None else torch.empty(0) for a in args], Z)
        ctx.has_affine = (q is not None, r is not None, qf is not None)
        ctx.dims = (n, m, N, b, flags)
        ctx.mark_non_differentiable(info)
        body = Z[:, :(N - 1) * (n + m)].view(b, N - 1, n + m)
        X = torch.cat([body[:, :, :n], Z[:, None, (N - 1) * (n + m):]], dim=1)
        return X, body[:, :, n:].contiguous(), info

    @staticmethod
    @once_differentiable  # double backward is not provided: create_graph=True raises instead of returning constants
    def backward(ctx, dX, dU, _dinfo):
        n, m, N, b, flags = ctx.dims
        A, B, Q, R, q, r, Qf, qf, Z = ctx.saved_tensors
        q, r, qf = (a if has else None for a, has in zip((q, r, qf), ctx.has_affine))
        dZ = torch.zeros_like(Z)
        body = dZ[:, :(N - 1) * (n + m)].view(b, N - 1, n + m)
        if dX is not None:
            body[:, :, :n] = dX[:, :N - 1]
            dZ[:, (N - 1) * (n + m):] = dX[:, N - 1]
        if dU is not None:
            body[:, :, n:] = dU
        want = ctx.needs_input_grad[1:]
        if not any(want):
            return (None,) * 10
        like = (A, B, Q, R, q, r, Qf, qf, Z.new_empty(b, n))  # an absent q, r, qf needs no gradient
        g = [torch.empty_like(t) if w else None for t, w in zip(like, want)]
        with torch.cuda.device(Z.device):
            ops.riccati_grad(_handle(Z.device), n, m, N, b, flags, A, B, Q, R, q, r, Qf, qf, Z, dZ, *g)
        for i in (0, 1, 2, 3, 6):  # column-major buffers -> math order
            if g[i] is not None:
                g[i] = g[i].transpose(-1, -2)
        return (None, *g)


def riccati_solve(A, B, Q, R, q, r, Qf, qf, x0, N: int | None = None):
    """Differentiable batched LQR solve; see the module docstring."""
    ts = [t for t in (A, B, Q, R, q, r, Qf, qf, x0) if t is not None]
    for t in ts:
        if not (t.is_cuda and t.dtype == torch.float64):
            raise TypeError("riccati_solve takes CUDA float64 tensors (there is no CPU path)")
    lti = A.dim() == 3
    if lti:
        if N is None:
            raise ValueError("an LTI problem (A of shape (b, n, n)) needs N")
    else:
        if N is not None and N != A.shape[1] + 1:
            raise ValueError(f"N = {N} does not match A's knot axis ({A.shape[1]})")
        N = A.shape[1] + 1
    b = max(t.shape[0] for t in ts)

    def full(t, sym=False):
        if t is None:
            return None
        if sym:
            t = 0.5 * (t + t.transpose(-1, -2))
        return t.expand((b,) + tuple(t.shape[1:])).contiguous()
    return _RiccatiSolve.apply(int(N), full(A), full(B), full(Q, True), full(R, True), full(q), full(r),
                               full(Qf, True), full(qf), full(x0))
