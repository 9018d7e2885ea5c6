"""Thin functional layer over the C ABI: every function takes raw buffers (numpy arrays for host
memory, torch CUDA tensors for device memory) already in the ABI's layouts and forwards the call.
No arithmetic happens here."""
from __future__ import annotations

import math

import numpy as np

from . import _lib
from ._lib import Handle, ptr

_default_handles: dict[int, Handle] = {}


def default_handle(device: int = 0) -> Handle:
    h = _default_handles.get(device)
    if h is None:
        h = _default_handles[device] = Handle(device)
    return h


def _p32(p):
    return np.ascontiguousarray(p, dtype=np.int32)


# ------------------------------------------------------------------ Riccati
def riccati(h: Handle, n, m, N, batch, flags, A, B, Q, R, q, r, Qf, qf, x0, Z, K=None, kff=None, info=None):
    """lqrb_riccati_f64: instance-major column-major buffers, host or device."""
    h.call("lqrb_riccati_f64", n, m, N, batch, flags, ptr(A), ptr(B), ptr(Q), ptr(R), ptr(q), ptr(r),
           ptr(Qf), ptr(qf), ptr(x0), ptr(Z), ptr(K), ptr(kff), ptr(info))


def riccati_grad(h: Handle, n, m, N, batch, flags, A, B, Q, R, q, r, Qf, qf, Z, dZ, gA=None, gB=None, gQ=None,
                 gR=None, gq=None, gr=None, gQf=None, gqf=None, gx0=None, info=None):
    """lqrb_riccati_grad_f64: gradients of l(Z) through lqrb_riccati_f64 from dZ = dl/dZ; buffers as riccati()."""
    h.call("lqrb_riccati_grad_f64", n, m, N, batch, flags, ptr(A), ptr(B), ptr(Q), ptr(R), ptr(q), ptr(r), ptr(Qf),
           ptr(qf), ptr(Z), ptr(dZ), ptr(gA), ptr(gB), ptr(gQ), ptr(gR), ptr(gq), ptr(gr), ptr(gQf), ptr(gqf), ptr(gx0),
           ptr(info))


def riccati_grad_gains(h: Handle, n, m, N, batch, flags, A, B, Q, R, q, r, Qf, qf, Z, dZ, dK, dkff, gA=None, gB=None,
                       gQ=None, gR=None, gq=None, gr=None, gQf=None, gqf=None, gx0=None, info=None):
    """lqrb_riccati_grad_gains_f64: gradients of l(Z, K, kff) through lqrb_riccati_f64 from the cotangents dZ, dK, dkff
    (each may be None, not all; Z only with dZ); buffers as riccati(), dK and dkff in the layout of its K, kff."""
    h.call("lqrb_riccati_grad_gains_f64", n, m, N, batch, flags, ptr(A), ptr(B), ptr(Q), ptr(R), ptr(q), ptr(r),
           ptr(Qf), ptr(qf), ptr(Z), ptr(dZ), ptr(dK), ptr(dkff), ptr(gA), ptr(gB), ptr(gQ), ptr(gR), ptr(gq), ptr(gr),
           ptr(gQf), ptr(gqf), ptr(gx0), ptr(info))


def riccati_pack(h: Handle, n, m, N, batch, flags, A, B, Q, R, q, r, Qf, qf, x0, knots, term):
    h.call("lqrb_riccati_pack_f64", n, m, N, batch, flags, ptr(A), ptr(B), ptr(Q), ptr(R), ptr(q), ptr(r),
           ptr(Qf), ptr(qf), ptr(x0), ptr(knots), ptr(term))


def riccati_solve_packed(h: Handle, n, m, N, batch, flags, knots, term, Z, gains=None, info=None):
    h.call("lqrb_riccati_solve_packed_f64", n, m, N, batch, flags, ptr(knots), ptr(term), ptr(Z),
           ptr(gains), ptr(info))


def riccati_tile_width(h: Handle, n, m) -> int:
    t = int(_lib.lib().lqrb_riccati_tile_width(h._h, n, m))
    if t <= 0:
        raise _lib.LqrbError(f"lqrb_riccati_tile_width: bad argument {-t}")
    return t


def riccati_unpack(h: Handle, n, m, N, batch, Zp, gains, Z, K=None, kff=None):
    """Packed outputs of riccati_solve_packed -> instance-major (applies the size class's tile width)."""
    h.call("lqrb_riccati_unpack_f64", n, m, N, batch, ptr(Zp), ptr(gains), ptr(Z), ptr(K), ptr(kff))


def unpack_rows(h: Handle, rows, batch, tile, packed, out):
    h.call("lqrb_unpack_rows_f64", rows, batch, tile, ptr(packed), ptr(out))


def pack_rows(h: Handle, rows, batch, tile, src, packed):
    h.call("lqrb_pack_rows_f64", rows, batch, tile, ptr(src), ptr(packed))


def rollout(h: Handle, n, m, N, batch, flags, A, B, x0, U, X):
    h.call("lqrb_rollout_f64", n, m, N, batch, flags, ptr(A), ptr(B), ptr(x0), ptr(U), ptr(X))


def lsq_solve(h: Handle, n, m, N, batch, A, B, Q, R, Qf, x0, Z, info=None):
    """lqrb_lsq_solve_f64: condensed least-squares solve of the LTI problem (src/least_squares.jl:158-190)."""
    h.call("lqrb_lsq_solve_f64", n, m, N, batch, ptr(A), ptr(B), ptr(Q), ptr(R), ptr(Qf), ptr(x0), ptr(Z), ptr(info))


# ------------------------------------------------------------------ BlockCholesky
def block_cholesky(h: Handle, n, m, batch, mode, A, B, C, M, info=None):
    h.call("lqrb_block_cholesky_f64", n, m, batch, mode, ptr(A), ptr(B), ptr(C), ptr(M), ptr(info))


def block_ldiv(h: Handle, n, m, batch, mode, M, nrhs, b):
    h.call("lqrb_block_ldiv_f64", n, m, batch, mode, ptr(M), nrhs, ptr(b))


# ------------------------------------------------------------------ KKT
def kkt_solve(h: Handle, n, m, N, batch, p, hess_mode, flags, Q, R, Hux, q, r, A, B, d, D2, C, c, dz, mult,
              res=None, info=None):
    p = _p32(p)
    h.call("lqrb_kkt_solve_f64", n, m, N, batch, p.ctypes.data, hess_mode, flags, ptr(Q), ptr(R), ptr(Hux),
           ptr(q), ptr(r), ptr(A), ptr(B), ptr(d), ptr(D2), ptr(C), ptr(c), ptr(dz), ptr(mult), ptr(res),
           ptr(info))


def kkt_grad(h: Handle, n, m, N, batch, p, hess_mode, flags, Q, R, Hux, A, B, D2, C, dz, mult, dz_bar, mult_bar,
             gQ=None, gR=None, gHux=None, gq=None, gr=None, gA=None, gB=None, gd=None, gD2=None, gC=None, gc=None,
             info=None):
    """lqrb_kkt_grad_f64: gradients of l(dz, mult) through lqrb_kkt_solve_f64 from the cotangents dz_bar, mult_bar;
    buffers as kkt_solve()."""
    p = _p32(p)
    h.call("lqrb_kkt_grad_f64", n, m, N, batch, p.ctypes.data, hess_mode, flags, ptr(Q), ptr(R), ptr(Hux), ptr(A),
           ptr(B), ptr(D2), ptr(C), ptr(dz), ptr(mult), ptr(dz_bar), ptr(mult_bar), ptr(gQ), ptr(gR), ptr(gHux),
           ptr(gq), ptr(gr), ptr(gA), ptr(gB), ptr(gd), ptr(gD2), ptr(gC), ptr(gc), ptr(info))


def kkt_pack(h: Handle, n, m, N, batch, p, hess_mode, Q, R, Hux, q, r, A, B, d, D2, C, c, data):
    p = _p32(p)
    h.call("lqrb_kkt_pack_f64", n, m, N, batch, p.ctypes.data, hess_mode, ptr(Q), ptr(R), ptr(Hux), ptr(q),
           ptr(r), ptr(A), ptr(B), ptr(d), ptr(D2), ptr(C), ptr(c), ptr(data))


def kkt_solve_packed(h: Handle, n, m, N, batch, p, hess_mode, explicit_d2, flags, data, dz, mult, res=None,
                     info=None):
    p = _p32(p)
    h.call("lqrb_kkt_solve_packed_f64", n, m, N, batch, p.ctypes.data, hess_mode, int(explicit_d2), flags,
           ptr(data), ptr(dz), ptr(mult), ptr(res), ptr(info))


def kkt_tile_width(h: Handle, n, m, N, p, hess_mode, explicit_d2=False) -> int:
    p = _p32(p)
    t = int(_lib.lib().lqrb_kkt_tile_width(h._h, n, m, N, p.ctypes.data, hess_mode, int(explicit_d2)))
    if t <= 0:
        raise _lib.LqrbError(f"lqrb_kkt_tile_width: bad argument {-t}")
    return t


def kkt_unpack(h: Handle, n, m, N, batch, p, hess_mode, explicit_d2, dzp, multp, resp, dz, mult, res=None):
    """Packed outputs of kkt_solve_packed -> instance-major (applies the shape's tile width)."""
    p = _p32(p)
    h.call("lqrb_kkt_unpack_f64", n, m, N, batch, p.ctypes.data, hess_mode, int(explicit_d2), ptr(dzp), ptr(multp),
           ptr(resp), ptr(dz), ptr(mult), ptr(res))


def kkt_factor(h: Handle, n, m, N, batch, p, hess_mode, flags, Q, R, Hux, A, B, D2, C, info=None):
    """calculate_shur_factors! (matrices) + cholesky!(U, F); the handle keeps the factor."""
    p = _p32(p)
    h.call("lqrb_kkt_factor_f64", n, m, N, batch, p.ctypes.data, hess_mode, flags, ptr(Q), ptr(R), ptr(Hux), ptr(A),
           ptr(B), ptr(D2), ptr(C), ptr(info))


def kkt_solve_factored(h: Handle, n, m, N, batch, p, hess_mode, explicit_d2, flags, q, r, d, c, dz, mult, res=None,
                       info=None):
    """forward / backward substitution + primals with the kept factor and a new right-hand side."""
    p = _p32(p)
    h.call("lqrb_kkt_solve_factored_f64", n, m, N, batch, p.ctypes.data, hess_mode, int(explicit_d2), flags, ptr(q),
           ptr(r), ptr(d), ptr(c), ptr(dz), ptr(mult), ptr(res), ptr(info))


def kkt_get_shur(h: Handle, n, m, N, batch, p, hess_mode, flags, Q, R, Hux, q, r, A, B, d, D2, C, c, S=None, hvec=None,
                 U=None, info=None):
    """dense S, h, U of the device's block rows (get_shur_factors / get_cholesky)."""
    p = _p32(p)
    h.call("lqrb_kkt_get_shur_f64", n, m, N, batch, p.ctypes.data, hess_mode, flags, ptr(Q), ptr(R), ptr(Hux), ptr(q),
           ptr(r), ptr(A), ptr(B), ptr(d), ptr(D2), ptr(C), ptr(c), ptr(S), ptr(hvec), ptr(U), ptr(info))


def kkt_residual(h: Handle, n, m, N, batch, p, flags, q, r, A, B, D2, C, mult, res=None, norms=None):
    """res_k = D1'lam_k + C'mu_k + D2'lam_{k-1} + g_k for given multipliers (residual, src/cholesky_solver.jl:238-252)."""
    p = _p32(p)
    h.call("lqrb_kkt_residual_f64", n, m, N, batch, p.ctypes.data, flags, ptr(q), ptr(r), ptr(A), ptr(B), ptr(D2),
           ptr(C), ptr(mult), ptr(res), ptr(norms))


# ------------------------------------------------------------------ layout helpers (host, numpy)
def cm(a):
    """math-order (..., rows, cols) -> column-major contiguous float64 buffer (Julia order)."""
    if a is None:
        return None
    return np.ascontiguousarray(np.swapaxes(np.asarray(a, dtype=np.float64), -1, -2))


def f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def kkt_flatten(prob: dict) -> dict:
    """math-order KKT problem dict (see problems.py) -> the ABI's instance-major column-major buffers."""
    n, m, N = prob["n"], prob["m"], prob["N"]
    b = prob["q"].shape[0]
    p = _p32(prob["p"])
    Cf = [np.swapaxes(np.asarray(Ck, dtype=np.float64), -1, -2).reshape(b, -1) for Ck in prob["C"]]
    cf = [np.asarray(ck, dtype=np.float64).reshape(b, -1) for ck in prob["c"]]
    Cflat = np.ascontiguousarray(np.concatenate(Cf, axis=1)) if Cf else np.zeros((b, 0))
    cflat = np.ascontiguousarray(np.concatenate(cf, axis=1)) if cf else np.zeros((b, 0))
    D2 = prob.get("D2")
    if D2 is not None:
        D2 = np.ascontiguousarray(np.concatenate(
            [np.swapaxes(np.asarray(x, dtype=np.float64), -1, -2).reshape(b, -1) for x in D2], axis=1))
    return dict(n=n, m=m, N=N, batch=b, p=p, hess_mode=int(prob.get("hess_mode", _lib.HESS_BLOCKDIAG)),
                Q=cm(prob["Q"]), R=cm(prob["R"]), Hux=cm(prob.get("Hux")), q=f64(prob["q"]), r=f64(prob["r"]),
                A=cm(prob["A"]), B=cm(prob["B"]), d=f64(prob["d"]), D2=D2, C=Cflat, c=cflat)


def kkt_solve_problem(prob: dict, soc: bool = False, want_res: bool = False, handle: Handle | None = None):
    """Solve a (math-order or flattened) KKT problem dict from host memory.
    Returns dz (b,NN), mult (b,P), info (b,)[, res (b,NN)]."""
    h = handle or default_handle()
    f = prob if "batch" in prob else kkt_flatten(prob)
    n, m, N, b = f["n"], f["m"], f["N"], f["batch"]
    NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, f["p"])
    dz, mult = np.zeros((b, NN)), np.zeros((b, P))
    res = np.zeros((b, NN)) if want_res else None
    info = np.zeros(b, dtype=np.int32)
    kkt_solve(h, n, m, N, b, f["p"], f["hess_mode"], _lib.FLAG_SOC if soc else 0, f["Q"], f["R"], f["Hux"],
              f["q"], f["r"], f["A"], f["B"], f["d"], f["D2"], f["C"], f["c"], dz, mult, res, info)
    return (dz, mult, info, res) if want_res else (dz, mult, info)


def kkt_grad_problem(prob: dict, dz, mult, dz_bar, mult_bar, handle: Handle | None = None):
    """Gradients of l(dz, mult) through the solve of a math-order KKT problem dict, from host memory.  dz (b, NN) and
    mult (b, P) are the outputs of the solve, dz_bar and mult_bar the cotangents of the same shapes (either may be
    None).  Returns (grads, info): grads holds math-order arrays with the shapes of the problem's Q, R, Hux, q, r, A,
    B, d, D2, C, c (keys likewise; D2, C, c are per-knot lists, Hux and D2 None where the problem has none)."""
    h = handle or default_handle()
    f = kkt_flatten(prob)
    n, m, N, b, p, mode = f["n"], f["m"], f["N"], f["batch"], f["p"], f["hess_mode"]
    dense = mode == _lib.HESS_DENSE
    g = dict(Q=np.zeros((b, N, n, n)), R=np.zeros((b, N - 1, m, m)), Hux=np.zeros((b, N - 1, n, m)) if dense else None,
             q=np.zeros((b, N, n)), r=np.zeros((b, N - 1, m)), A=np.zeros((b, N - 1, n, n)),
             B=np.zeros((b, N - 1, m, n)), d=np.zeros((b, N - 1, n)),
             D2=np.zeros_like(f["D2"]) if f["D2"] is not None else None,
             C=np.zeros_like(f["C"]) if f["C"].shape[1] else None, c=np.zeros_like(f["c"]) if f["c"].shape[1] else None)
    info = np.zeros(b, dtype=np.int32)
    kkt_grad(h, n, m, N, b, p, mode, 0, f["Q"], f["R"], f["Hux"], f["A"], f["B"], f["D2"], f["C"], f64(dz), f64(mult),
             f64(dz_bar), f64(mult_bar), g["Q"], g["R"], g["Hux"], g["q"], g["r"], g["A"], g["B"], g["d"], g["D2"],
             g["C"], g["c"], info)
    for k in ("Q", "R", "Hux", "A", "B"):  # column-major buffers -> math order
        if g[k] is not None:
            g[k] = np.ascontiguousarray(np.swapaxes(g[k], -1, -2))
    ws = [n + (m if k < N - 1 else 0) for k in range(N)]
    if g["D2"] is not None:  # blocks n x w_k, k = 2..N
        cuts = np.cumsum([n * w for w in ws[1:]])[:-1]
        g["D2"] = [np.swapaxes(x.reshape(b, w, n), -1, -2).copy() for x, w in zip(np.split(g["D2"], cuts, axis=1), ws[1:])]
    Cf = g["C"] if g["C"] is not None else np.zeros((b, 0))
    cf = g["c"] if g["c"] is not None else np.zeros((b, 0))
    Cs = np.split(Cf, np.cumsum([int(pk) * w for pk, w in zip(p, ws)])[:-1], axis=1)
    g["C"] = [np.swapaxes(x.reshape(b, w, int(pk)), -1, -2).copy() for x, w, pk in zip(Cs, ws, p)]
    g["c"] = [x.copy() for x in np.split(cf, np.cumsum(p)[:-1], axis=1)]
    return g, info


def riccati_flatten(prob: dict) -> dict:
    return dict(n=prob["n"], m=prob["m"], N=prob["N"], lti=bool(prob.get("lti", False)),
                batch=prob["x0"].shape[0], A=cm(prob["A"]), B=cm(prob["B"]), Q=cm(prob["Q"]), R=cm(prob["R"]),
                q=f64(prob.get("q")), r=f64(prob.get("r")), Qf=cm(prob["Qf"]), qf=f64(prob.get("qf")),
                x0=f64(prob["x0"]))


def riccati_solve_problem(prob: dict, want_gains: bool = True, handle: Handle | None = None):
    """Solve a Riccati problem dict from host memory.
    Returns X (b,N,n), U (b,N-1,m), K (b,N-1,m,n), kff (b,N-1,m), info."""
    h = handle or default_handle()
    f = prob if "batch" in prob else riccati_flatten(prob)
    n, m, N, b = f["n"], f["m"], f["N"], f["batch"]
    NN = _lib.num_vars(n, m, N)
    Z = np.zeros((b, NN))
    K = np.zeros((b, N - 1, n, m)) if want_gains else None
    kff = np.zeros((b, N - 1, m)) if want_gains else None
    info = np.zeros(b, dtype=np.int32)
    riccati(h, n, m, N, b, _lib.FLAG_LTI if f["lti"] else 0, f["A"], f["B"], f["Q"], f["R"], f["q"], f["r"],
            f["Qf"], f["qf"], f["x0"], Z, K, kff, info)
    X, U = split_primals(Z, n, m, N)
    return X, U, (np.swapaxes(K, -1, -2).copy() if want_gains else None), kff, info


def riccati_grad_problem(prob: dict, Z, dZ, handle: Handle | None = None):
    """Gradients of l(Z) through the solve of a Riccati problem dict, from host memory.  Z is the (b, NN) Primals
    output of the solve and dZ = dl/dZ of the same shape.  Returns (grads, info): grads holds math-order arrays with
    the shapes of the problem's A, B, Q, R, q, r, Qf, qf, x0 (keys likewise)."""
    h = handle or default_handle()
    f = prob if "batch" in prob else riccati_flatten(prob)
    n, m, N, b = f["n"], f["m"], f["N"], f["batch"]
    kn = (b,) if f["lti"] else (b, N - 1)
    g = dict(A=np.zeros(kn + (n, n)), B=np.zeros(kn + (m, n)), Q=np.zeros(kn + (n, n)), R=np.zeros(kn + (m, m)),
             q=np.zeros(kn + (n,)), r=np.zeros(kn + (m,)), Qf=np.zeros((b, n, n)), qf=np.zeros((b, n)),
             x0=np.zeros((b, n)))
    info = np.zeros(b, dtype=np.int32)
    riccati_grad(h, n, m, N, b, _lib.FLAG_LTI if f["lti"] else 0, f["A"], f["B"], f["Q"], f["R"], f["q"], f["r"],
                 f["Qf"], f["qf"], f64(Z), f64(dZ), g["A"], g["B"], g["Q"], g["R"], g["q"], g["r"], g["Qf"], g["qf"],
                 g["x0"], info)
    for k in ("A", "B", "Q", "R", "Qf"):  # column-major buffers -> math order
        g[k] = np.ascontiguousarray(np.swapaxes(g[k], -1, -2))
    return g, info


def riccati_grad_gains_problem(prob: dict, Z, dZ, dK, dkff, handle: Handle | None = None):
    """Gradients of l(Z, K, kff) through the solve of a Riccati problem dict, from host memory.  Z is the (b, NN)
    Primals output of the solve, dZ = dl/dZ of the same shape, dK = dl/dK (b, N-1, m, n) and dkff = dl/dkff (b, N-1, m)
    in math order; each cotangent may be None, not all (Z only with dZ).  Returns (grads, info) as
    riccati_grad_problem."""
    h = handle or default_handle()
    f = prob if "batch" in prob else riccati_flatten(prob)
    n, m, N, b = f["n"], f["m"], f["N"], f["batch"]
    kn = (b,) if f["lti"] else (b, N - 1)
    g = dict(A=np.zeros(kn + (n, n)), B=np.zeros(kn + (m, n)), Q=np.zeros(kn + (n, n)), R=np.zeros(kn + (m, m)),
             q=np.zeros(kn + (n,)), r=np.zeros(kn + (m,)), Qf=np.zeros((b, n, n)), qf=np.zeros((b, n)),
             x0=np.zeros((b, n)))
    info = np.zeros(b, dtype=np.int32)
    riccati_grad_gains(h, n, m, N, b, _lib.FLAG_LTI if f["lti"] else 0, f["A"], f["B"], f["Q"], f["R"], f["q"], f["r"],
                       f["Qf"], f["qf"], f64(Z), f64(dZ), cm(dK), f64(dkff), g["A"], g["B"], g["Q"], g["R"], g["q"],
                       g["r"], g["Qf"], g["qf"], g["x0"], info)
    for k in ("A", "B", "Q", "R", "Qf"):  # column-major buffers -> math order
        g[k] = np.ascontiguousarray(np.swapaxes(g[k], -1, -2))
    return g, info


def dare(h: Handle, n, m, batch, A, B, Q, R, P=None, K=None, iters=None, info=None):
    """lqrb_dare_f64: stabilising solution P [n,n,batch] and gain K [m,n,batch] of the discrete algebraic Riccati
    equation; instance-major column-major buffers, host or device."""
    h.call("lqrb_dare_f64", n, m, batch, ptr(A), ptr(B), ptr(Q), ptr(R), ptr(P), ptr(K), ptr(iters), ptr(info))


def dare_grad(h: Handle, n, m, batch, A, B, R, P, dP, dK, gA=None, gB=None, gQ=None, gR=None, info=None):
    """lqrb_dare_grad_f64: gradients of l(P, K) through lqrb_dare_f64 from dP = dl/dP, dK = dl/dK (either may be
    None, not both); buffers as dare()."""
    h.call("lqrb_dare_grad_f64", n, m, batch, ptr(A), ptr(B), ptr(R), ptr(P), ptr(dP), ptr(dK), ptr(gA), ptr(gB),
           ptr(gQ), ptr(gR), ptr(info))


def dare_problem(prob: dict, handle: Handle | None = None):
    """Solve the DARE of the math-order arrays A (b,n,n), B (b,n,m), Q (b,n,n), R (b,m,m) of a problem dict (an LTI
    Riccati problem dict serves) from host memory.  Returns P (b,n,n), K (b,m,n), iters (b,), info (b,)."""
    h = handle or default_handle()
    A, B = np.asarray(prob["A"]), np.asarray(prob["B"])
    b, n, m = A.shape[0], A.shape[-1], B.shape[-1]
    P, K = np.zeros((b, n, n)), np.zeros((b, n, m))  # column-major buffers
    iters, info = np.zeros(b, dtype=np.int32), np.zeros(b, dtype=np.int32)
    dare(h, n, m, b, cm(A), cm(B), cm(prob["Q"]), cm(prob["R"]), P, K, iters, info)
    return np.swapaxes(P, -1, -2).copy(), np.swapaxes(K, -1, -2).copy(), iters, info


def dare_grad_problem(prob: dict, P, dP=None, dK=None, handle: Handle | None = None):
    """Gradients of l(P, K) through dare_problem, from host memory: P (b,n,n) as it returned, dP = dl/dP (b,n,n),
    dK = dl/dK (b,m,n) in math order (either may be None, not both).  Returns (grads, info): grads holds math-order
    arrays A, B, Q, R with the shapes of the problem's."""
    h = handle or default_handle()
    A, B = np.asarray(prob["A"]), np.asarray(prob["B"])
    b, n, m = A.shape[0], A.shape[-1], B.shape[-1]
    g = dict(A=np.zeros((b, n, n)), B=np.zeros((b, m, n)), Q=np.zeros((b, n, n)), R=np.zeros((b, m, m)))
    info = np.zeros(b, dtype=np.int32)
    dare_grad(h, n, m, b, cm(A), cm(B), cm(prob["R"]), cm(P), cm(dP), cm(dK), g["A"], g["B"], g["Q"], g["R"], info)
    return {k: np.ascontiguousarray(np.swapaxes(v, -1, -2)) for k, v in g.items()}, info


def admm_cache_doubles(n, m) -> int:
    """doubles per instance of the lqrb_admm_cache_f64 record [A | B | Q | R | Qf | K | C1 | C2 | rho]"""
    return 4 * n * n + 2 * n * m + 2 * m * m + 1


def admm_cache_split(cache, n, m) -> dict:
    """(b, L) cache records -> dict of math-order views A, B, Q, R, Qf, K, C1, C2 (b, rows, cols) and rho (b,)"""
    out, o = {}, 0
    for k, (r, c) in zip(("A", "B", "Q", "R", "Qf", "K", "C1", "C2"),
                         ((n, n), (n, m), (n, n), (m, m), (n, n), (m, n), (m, m), (n, n))):
        out[k] = cache[:, o:o + r * c].reshape(-1, c, r).swapaxes(-1, -2)
        o += r * c
    out["rho"] = cache[:, o]
    return out


def admm_cache(h: Handle, n, m, batch, rho, A, B, Q, R, cache, info=None):
    """lqrb_admm_cache_f64: the ADMM cache of (A, B, Q, R, rho); instance-major column-major buffers, host or device."""
    h.call("lqrb_admm_cache_f64", n, m, batch, float(rho), ptr(A), ptr(B), ptr(Q), ptr(R), ptr(cache), ptr(info))


def admm_solve(h: Handle, n, m, N, batch, cache, x0, Z, xref=None, uref=None, umin=None, umax=None, xmin=None,
               xmax=None, state=None, warm=False, max_iter=100, eps_pri=1e-6, eps_dual=1e-6, iters=None, res=None,
               info=None):
    """lqrb_admm_solve_f64: box-constrained MPC by ADMM on a cache from admm_cache(); buffers as in the header
    (instance-major column-major, host or device); `state` is updated in place, read when `warm`."""
    o = _lib.AdmmOptions(max_iter=int(max_iter), eps_pri=float(eps_pri), eps_dual=float(eps_dual))
    import ctypes as C
    h.call("lqrb_admm_solve_f64", n, m, N, batch, _lib.FLAG_WARM_START if warm else 0, C.byref(o), ptr(cache), ptr(x0),
           ptr(xref), ptr(uref), ptr(umin), ptr(umax), ptr(xmin), ptr(xmax), ptr(state), ptr(Z), ptr(iters), ptr(res),
           ptr(info))


def admm_cache_problem(prob: dict, rho, handle: Handle | None = None):
    """The ADMM cache of the math-order arrays A (b,n,n), B (b,n,m), Q (b,n,n), R (b,m,m) of a problem dict (an LTI
    Riccati problem dict serves), from host memory.  Returns (cache (b, L), info (b,)); admm_cache_split() reads it."""
    h = handle or default_handle()
    A, B = np.asarray(prob["A"]), np.asarray(prob["B"])
    b, n, m = A.shape[0], A.shape[-1], B.shape[-1]
    cache = np.zeros((b, admm_cache_doubles(n, m)))
    info = np.zeros(b, dtype=np.int32)
    admm_cache(h, n, m, b, rho, cm(A), cm(B), cm(prob["Q"]), cm(prob["R"]), cache, info)
    return cache, info


def admm_solve_problem(cache, x0, N, xref=None, uref=None, umin=None, umax=None, xmin=None, xmax=None, state=None,
                       warm=False, max_iter=100, eps_pri=1e-6, eps_dual=1e-6, handle: Handle | None = None):
    """lqrb_admm_solve_f64 from host memory on math-order arrays: cache (b, L), x0 (b,n), xref (b,N,n), uref (b,N-1,m),
    umin / umax (b,N-1,m), xmin / xmax (b,N-1,n), each optional; state (b, 2(N-1)(m+n)) is updated in place when given.
    Returns X (b,N,n), U (b,N-1,m), iters (b,), res (b,2), info (b,)."""
    h = handle or default_handle()
    x0 = f64(x0)
    b, n = x0.shape
    m = (math.isqrt(n * n + 2 * (cache.shape[1] - 1 - 4 * n * n)) - n) // 2  # the root of 2m^2 + 2nm = L - 1 - 4n^2
    Z = np.zeros((b, _lib.num_vars(n, m, N)))
    iters, res, info = np.zeros(b, dtype=np.int32), np.zeros((b, 2)), np.zeros(b, dtype=np.int32)
    admm_solve(h, n, m, N, b, f64(cache), x0, Z, f64(xref), f64(uref), f64(umin), f64(umax), f64(xmin), f64(xmax),
               state, warm, max_iter, eps_pri, eps_dual, iters, res, info)
    X, U = split_primals(Z, n, m, N)
    return X, U, iters, res, info


def split_primals(Z, n, m, N):
    """Primals layout [x1;u1;...;xN] (src/lqr_problem.jl:46-73) -> X (b,N,n), U (b,N-1,m) copies."""
    b = Z.shape[0]
    body = Z[:, :(N - 1) * (n + m)].reshape(b, N - 1, n + m)
    X = np.concatenate([body[:, :, :n], Z[:, None, (N - 1) * (n + m):]], axis=1)
    return X, body[:, :, n:].copy()


# ------------------------------------------------------------------ Dubins SQP
def sqp_dubins(h: Handle, batch, opts: dict, x0, xf, Z, feas_p=None, feas_d=None, iters=None):
    """lqrb_sqp_dubins_f64; Z is updated in place.  Returns the total number of KKT solves."""
    import ctypes as C
    o = _lib.SqpOptions(N=int(opts["N"]), iters=int(opts["iters"]), dt=float(opts["dt"]),
                        q_diag=float(opts["q_diag"]), r_diag=float(opts["r_diag"]), qf_diag=float(opts["qf_diag"]),
                        eps_p=float(opts.get("eps_p", 1e-5)), eps_d=float(opts.get("eps_d", 1e-5)),
                        line_search=int(opts.get("line_search", 1)))
    solves = C.c_int64(0)
    h.call("lqrb_sqp_dubins_f64", batch, C.byref(o), ptr(x0), ptr(xf), ptr(Z), ptr(feas_p), ptr(feas_d), ptr(iters),
           C.byref(solves))
    return int(solves.value)
