"""Differentiable batched Riccati and constrained KKT solves for torch (``lqr_b200.autograd``).

``riccati_solve(A, B, Q, R, q, r, Qf, qf, x0, N=None) -> (X, U, info)`` solves the LTV-affine LQR of
``lqrb_riccati_f64`` on CUDA float64 tensors in math order and backpropagates through it with
``lqrb_riccati_grad_f64``: the adjoint of an LQR is another LQR with the same matrices, so the backward pass is one
more solve on the same kernels plus one sweep that forms the gradients.  With ``gains=True`` it returns
``(X, U, K, kff, info)``, the policy u_k = -K_k x_k - kff_k included (K (b, N-1, m, n), kff (b, N-1, m)), and
backpropagates through all four outputs with ``lqrb_riccati_grad_gains_f64``.

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

``kkt_solve(Q, R, q, r, A, B, d, C, c, Hux=None, D2=None, hess_mode=HESS_BLOCKDIAG) -> (X, U, mult, info)`` solves the
constrained KKT system of ``lqrb_kkt_solve_f64`` and backpropagates through it with ``lqrb_kkt_grad_f64``: one more
solve of the same KKT matrices with the cotangents as right-hand side, then one kernel that forms the gradients.

Shapes (math order, batch first):
    Q (b, N, n, n)  R (b, N-1, m, m)  q (b, N, n)  r (b, N-1, m)  A (b, N-1, n, n)  B (b, N-1, n, m)  d (b, N-1, n)
    C, c: lists of N tensors C_k (b, p_k, w_k), c_k (b, p_k) with w_k = n + m (w_N = n); p is read from their shapes
    Hux (b, N-1, m, n) (LQRB_HESS_DENSE)   D2: None (D2_k = [-I 0]) or a list of N-1 tensors (b, n, w_k), k = 2..N
    ->  X (b, N, n), U (b, N-1, m), mult (b, P) in the order [mu_1; lam_1; ...; mu_N], info (b,) int32
Batch broadcasting, the symmetrisation of Q and R (under HESS_DIAG only their diagonals are read and receive gradient),
``info``, streams and the CPU rule are as for ``riccati_solve``.

``dare_solve(A, B, Q, R) -> (P, K, info)`` solves the discrete algebraic Riccati equation of the infinite-horizon LQR
with ``lqrb_dare_f64`` (structured doubling) and backpropagates through P and K with ``lqrb_dare_grad_f64`` (one Stein
equation).  A (b, n, n), B (b, n, m), Q (b, n, n), R (b, m, m)  ->  P (b, n, n), K (b, m, n) with u = -K x, info (b,)
int32 (0 ok, otherwise the codes of include/lqrb200.h; a failed instance's P, K and gradients are NaN).  Batch
broadcasting, the symmetrisation of Q and R, streams and the CPU rule are as for ``riccati_solve``; a loss on P alone or
K alone skips the other's cotangent.  ``riccati_solve(A, B, Q, R, q, r, Qf=P, qf, x0, N=N)`` with the same A, B, Q, R
composes with it into a finite-horizon MPC layer whose terminal cost is the infinite-horizon cost-to-go: its gains are
then K at every knot, and gradients flow through P into the stage-cost and dynamics arguments.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from . import _lib, ops

__all__ = ["riccati_solve", "kkt_solve", "dare_solve"]


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
    def forward(ctx, N, A, B, Q, R, q, r, Qf, qf, x0, gains=False):
        b, n, m = x0.shape[0], A.shape[-1], B.shape[-1]
        flags = _lib.FLAG_LTI if A.dim() == 3 else 0
        args = [_cm(A), _cm(B), _cm(Q), _cm(R), q, r, _cm(Qf), qf]
        Z = torch.empty(b, _lib.num_vars(n, m, N), dtype=torch.float64, device=x0.device)
        info = torch.empty(b, dtype=torch.int32, device=x0.device)
        K = torch.empty(b, N - 1, n, m, dtype=torch.float64, device=x0.device) if gains else None  # column-major m x n
        kff = torch.empty(b, N - 1, m, dtype=torch.float64, device=x0.device) if gains else None
        with torch.cuda.device(x0.device):
            ops.riccati(_handle(x0.device), n, m, N, b, flags, *args, x0, Z, K, kff, info)
        ctx.save_for_backward(*[a if a is not None else torch.empty(0) for a in args], Z)
        ctx.has_affine = (q is not None, r is not None, qf is not None)
        ctx.dims = (n, m, N, b, flags)
        ctx.gains = gains
        ctx.mark_non_differentiable(info)
        body = Z[:, :(N - 1) * (n + m)].view(b, N - 1, n + m)
        X = torch.cat([body[:, :, :n], Z[:, None, (N - 1) * (n + m):]], dim=1)
        if gains:
            ctx.set_materialize_grads(False)  # an unused output's cotangent stays None and costs no work
            return X, body[:, :, n:].contiguous(), K.transpose(-1, -2), kff, info
        return X, body[:, :, n:].contiguous(), info

    @staticmethod
    @once_differentiable  # double backward is not provided: create_graph=True raises instead of returning constants
    def backward(ctx, dX, dU, *rest):
        n, m, N, b, flags = ctx.dims
        A, B, Q, R, q, r, Qf, qf, Z = ctx.saved_tensors
        q, r, qf = (a if has else None for a, has in zip((q, r, qf), ctx.has_affine))
        dK, dkff = rest[:2] if ctx.gains else (None, None)
        want = ctx.needs_input_grad[1:10]
        if not any(want) or (ctx.gains and dX is None and dU is None and dK is None and dkff is None):
            return (None,) * 11
        dZ = None
        if not ctx.gains or dX is not None or dU is not None:
            dZ = torch.zeros_like(Z)
            body = dZ[:, :(N - 1) * (n + m)].view(b, N - 1, n + m)
            if dX is not None:
                body[:, :, :n] = dX[:, :N - 1]
                dZ[:, (N - 1) * (n + m):] = dX[:, N - 1]
            if dU is not None:
                body[:, :, n:] = dU
        like = (A, B, Q, R, q, r, Qf, qf, Z.new_empty(b, n))  # an absent q, r, qf needs no gradient
        g = [torch.empty_like(t) if w else None for t, w in zip(like, want)]
        with torch.cuda.device(Z.device):
            if ctx.gains:
                ops.riccati_grad_gains(_handle(Z.device), n, m, N, b, flags, A, B, Q, R, q, r, Qf, qf, Z, dZ,
                                       None if dK is None else _cm(dK), None if dkff is None else dkff.contiguous(),
                                       *g)
            else:
                ops.riccati_grad(_handle(Z.device), n, m, N, b, flags, A, B, Q, R, q, r, Qf, qf, Z, dZ, *g)
        for i in (0, 1, 2, 3, 6):  # column-major buffers -> math order
            if g[i] is not None:
                g[i] = g[i].transpose(-1, -2)
        return (None, *g, None)


def riccati_solve(A, B, Q, R, q, r, Qf, qf, x0, N: int | None = None, gains: bool = False):
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
                               full(Qf, True), full(qf), full(x0), bool(gains))


class _KktSolve(torch.autograd.Function):
    """On the ABI's instance-major buffers (column-major blocks, ragged arrays concatenated): kkt_solve lays the
    arguments out with differentiable torch operations, so the gradients of this function need no reshaping."""

    @staticmethod
    def forward(ctx, dims, p, Q, R, Hux, q, r, A, B, d, D2, C, c):
        n, m, N, b, hess = dims
        dz = torch.empty(b, _lib.num_vars(n, m, N), dtype=torch.float64, device=Q.device)
        mult = torch.empty(b, _lib.num_cons(n, N, p), dtype=torch.float64, device=Q.device)
        info = torch.empty(b, dtype=torch.int32, device=Q.device)
        with torch.cuda.device(Q.device):
            ops.kkt_solve(_handle(Q.device), n, m, N, b, p, hess, 0, Q, R, Hux, q, r, A, B, d, D2, C, c, dz, mult,
                          None, info)
        ctx.save_for_backward(*[a if a is not None else torch.empty(0) for a in (Q, R, Hux, A, B, D2, C)], dz, mult)
        ctx.absent = (Hux is None, D2 is None)
        ctx.shapes = [None if t is None else t.shape for t in (Q, R, Hux, q, r, A, B, d, D2, C, c)]
        ctx.dims, ctx.p = dims, p
        ctx.mark_non_differentiable(info)
        return dz, mult, info

    @staticmethod
    @once_differentiable  # double backward is not provided: create_graph=True raises instead of returning constants
    def backward(ctx, ddz, dmult, _dinfo):
        n, m, N, b, hess = ctx.dims
        Q, R, Hux, A, B, D2, C, dz, mult = ctx.saved_tensors
        Hux, D2 = (None if gone else t for t, gone in zip((Hux, D2), ctx.absent))
        rows = C.shape[1] > 0
        # an absent input, Hux outside LQRB_HESS_DENSE and C, c without stage rows get no gradient
        have = [s is not None for s in ctx.shapes]
        have[2] = have[2] and hess == _lib.HESS_DENSE
        have[9] = have[10] = rows
        g = [dz.new_empty(s) if (w and h) else None for s, w, h in zip(ctx.shapes, ctx.needs_input_grad[2:], have)]
        if all(x is None for x in g) or (ddz is None and dmult is None):
            return (None,) * 13
        with torch.cuda.device(dz.device):
            ops.kkt_grad(_handle(dz.device), n, m, N, b, ctx.p, hess, 0, Q, R, Hux, A, B, D2, C if rows else None, dz,
                         mult, ddz.contiguous() if ddz is not None else None,
                         dmult.contiguous() if dmult is not None else None, *g)
        return (None, None, *g)


def kkt_solve(Q, R, q, r, A, B, d, C, c, Hux=None, D2=None, hess_mode=_lib.HESS_BLOCKDIAG):
    """Differentiable batched constrained KKT solve; see the module docstring."""
    C, c, D2 = list(C), list(c), (None if D2 is None else list(D2))
    ts = [Q, R, q, r, A, B, d, *C, *c] + ([Hux] if Hux is not None else []) + (D2 or [])
    for t in ts:
        if not (t.is_cuda and t.dtype == torch.float64):
            raise TypeError("kkt_solve takes CUDA float64 tensors (there is no CPU path)")
    N, n, m = Q.shape[1], Q.shape[-1], R.shape[-1]
    if len(C) != N or len(c) != N or (D2 is not None and len(D2) != N - 1):
        raise ValueError("C and c need N blocks, D2 N-1")
    p = [int(Ck.shape[-2]) for Ck in C]
    b = max(t.shape[0] for t in ts)

    def full(t, sym=False):
        if sym:
            t = 0.5 * (t + t.transpose(-1, -2))
        return t.expand((b,) + tuple(t.shape[1:]))

    def flat(blocks):  # per-knot math-order blocks -> the ABI's concatenation of column-major blocks
        return torch.cat([_cm(full(x)).reshape(b, -1) for x in blocks], dim=1).contiguous()
    dz, mult, info = _KktSolve.apply(
        (n, m, N, b, int(hess_mode)), p, _cm(full(Q, True)), _cm(full(R, True)),
        None if Hux is None else _cm(full(Hux)), full(q).contiguous(), full(r).contiguous(), _cm(full(A)),
        _cm(full(B)), full(d).contiguous(), None if D2 is None else flat(D2), flat(C),
        torch.cat([full(x) for x in c], dim=1).contiguous())
    body = dz[:, :(N - 1) * (n + m)].view(b, N - 1, n + m)
    X = torch.cat([body[:, :, :n], dz[:, None, (N - 1) * (n + m):]], dim=1)
    return X, body[:, :, n:].contiguous(), mult, info


class _DareSolve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, A, B, Q, R):
        b, n, m = A.shape[0], A.shape[-1], B.shape[-1]
        Ac, Bc, Rc = _cm(A), _cm(B), _cm(R)
        P = torch.empty(b, n, n, dtype=torch.float64, device=A.device)  # symmetric: either order
        K = torch.empty(b, n, m, dtype=torch.float64, device=A.device)  # column-major m x n
        info = torch.empty(b, dtype=torch.int32, device=A.device)
        with torch.cuda.device(A.device):
            ops.dare(_handle(A.device), n, m, b, Ac, Bc, _cm(Q), Rc, P, K, None, info)
        ctx.save_for_backward(Ac, Bc, Rc, P)
        ctx.dims = (n, m, b)
        ctx.mark_non_differentiable(info)
        ctx.set_materialize_grads(False)  # a loss on P alone or K alone passes no cotangent for the other
        return P, K.transpose(-1, -2), info

    @staticmethod
    @once_differentiable  # double backward is not provided: create_graph=True raises instead of returning constants
    def backward(ctx, dP, dK, _dinfo):
        A, B, R, P = ctx.saved_tensors
        n, m, b = ctx.dims
        if (dP is None and dK is None) or not any(ctx.needs_input_grad):
            return (None,) * 4
        like = (A, B, P, R)  # gA, gB, gQ, gR: column-major buffers of the inputs' shapes
        g = [torch.empty_like(t) if w else None for t, w in zip(like, ctx.needs_input_grad)]
        with torch.cuda.device(A.device):
            ops.dare_grad(_handle(A.device), n, m, b, A, B, R, P, None if dP is None else _cm(dP),
                          None if dK is None else _cm(dK), *g)
        return tuple(None if x is None else x.transpose(-1, -2) for x in g)


def dare_solve(A, B, Q, R):
    """Differentiable batched DARE solve; see the module docstring."""
    for t in (A, B, Q, R):
        if not (t.is_cuda and t.dtype == torch.float64):
            raise TypeError("dare_solve takes CUDA float64 tensors (there is no CPU path)")
    b = max(t.shape[0] for t in (A, B, Q, R))

    def full(t, sym=False):
        if sym:
            t = 0.5 * (t + t.transpose(-1, -2))
        return t.expand((b,) + tuple(t.shape[1:]))
    return _DareSolve.apply(full(A), full(B), full(Q, True), full(R, True))
