"""Thin functional layer over the C ABI: every function takes raw buffers (numpy arrays for host
memory, torch CUDA tensors for device memory) already in the ABI's layouts and forwards the call.
No arithmetic happens here."""
from __future__ import annotations

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
