"""GPU: host and device arrays give the same results.  Every entry point that takes instance-major arrays runs once
with numpy arrays (staged through the device) and once with torch CUDA tensors (device-resident); the outputs and
`info` must be equal bit for bit.  The chunked entry points are also run in several host chunks, so that both copy
streams and their scratch are in use, and with host and device arrays mixed in one call."""
import numpy as np
import pytest

from lqr_b200 import _lib, ops, problems

pytestmark = pytest.mark.gpu

HOST, DEV = "host", "device"
DEV_INFO_HOST = "device, info on the host"   # an output kind: every output in device memory except `info`


def _to(kind, a):
    """numpy array -> the same values in host (numpy) or device (torch) memory."""
    if a is None or kind == HOST:
        return None if a is None else np.ascontiguousarray(a)
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _outs(kind, **spec):
    """Zeroed outputs {name: (shape, dtype)} in memory of the given kind."""
    def where(name):
        return (HOST if name == "info" else DEV) if kind == DEV_INFO_HOST else kind
    return {k: _to(where(k), np.zeros(shape, dtype=dt)) for k, (shape, dt) in spec.items()}


F8, I4 = np.float64, np.int32


def _np(a):
    return a if isinstance(a, np.ndarray) else a.cpu().numpy()


def _call(handle, fn, *args, **out):
    """fn(handle, *args, **out) once torch has finished writing the arguments; returns the outputs as numpy arrays."""
    import torch
    torch.cuda.synchronize()
    ret = fn(handle, *args, **out)
    handle.synchronize()
    return ret, {k: _np(v) for k, v in out.items()}


# ------------------------------------------------------------------ one case per entry point
# Each case takes the memory kind of its inputs and of its outputs and returns its outputs as numpy arrays.
def _riccati(handle, ik, ok, n=4, m=1, N=20, b=37):
    f = ops.riccati_flatten(problems.random_lqr_riccati(n, m, N, b, seed=11))
    names = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")
    L = _lib.riccati_layout(n, m, N)
    out = _outs(ok, Z=((b, L.z_rows), F8), K=((b, N - 1, n, m), F8), kff=((b, N - 1, m), F8), info=(b, I4))
    return _call(handle, ops.riccati, n, m, N, b, 0, *[_to(ik, f[k]) for k in names], **out)[1]


KKT_NAMES = ("Q", "R", "Hux", "q", "r", "A", "B", "d", "D2", "C", "c")


def _kkt_problem(n=12, m=4, N=10, b=37, mid_p=0):
    return ops.kkt_flatten(problems.random_lqr_kkt(n, m, N, b, seed=12, mid_p=mid_p, hess_mode=1))


def _kkt_solve(handle, ik, ok, f=None):
    f = f or _kkt_problem()
    n, m, N, b, p = f["n"], f["m"], f["N"], f["batch"], f["p"]
    NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
    out = _outs(ok, dz=((b, NN), F8), mult=((b, P), F8), res=((b, NN), F8), info=(b, I4))
    return _call(handle, ops.kkt_solve, n, m, N, b, p, f["hess_mode"], 0, *[_to(ik, f[k]) for k in KKT_NAMES], **out)[1]


def _kkt_residual(handle, ik, ok, f=None):
    f = f or _kkt_problem(n=5, m=2, N=12, b=37, mid_p=1)
    n, m, N, b, p = f["n"], f["m"], f["N"], f["batch"], f["p"]
    _, mult, _ = ops.kkt_solve_problem(f, handle=handle)
    NN = _lib.num_vars(n, m, N)
    out = _outs(ok, res=((b, NN), F8), norms=(b, F8))
    args = [_to(ik, f[k]) for k in ("q", "r", "A", "B", "D2", "C")] + [_to(ik, mult)]
    return _call(handle, ops.kkt_residual, n, m, N, b, p, 0, *args, **out)[1]


def _rollout(handle, ik, ok):
    n, m, N, b = 6, 3, 15, 37
    f = ops.riccati_flatten(problems.random_lqr_riccati(n, m, N, b, seed=13))
    U = np.random.default_rng(13).standard_normal((b, N - 1, m))
    args = [_to(ik, a) for a in (f["A"], f["B"], f["x0"], U)]
    return _call(handle, ops.rollout, n, m, N, b, 0, *args, **_outs(ok, X=((b, N, n), F8)))[1]


def _lsq(handle, ik, ok):
    n, m, N, b = 4, 1, 30, 9
    f = ops.riccati_flatten(problems.random_lqr_riccati(n, m, N, b, seed=14, lti=True))
    out = _outs(ok, Z=((b, _lib.num_vars(n, m, N)), F8), info=(b, I4))
    return _call(handle, ops.lsq_solve, n, m, N, b, *[_to(ik, f[k]) for k in ("A", "B", "Q", "R", "Qf", "x0")], **out)[1]


def _block_blocks(n=10, m=5, b=7):
    rng = np.random.default_rng(15)
    A = rng.random((b, n, n)); A = np.einsum("bki,bkj->bij", A, A)
    B = rng.random((b, m, m)); B = np.einsum("bki,bkj->bij", B, B)
    C = rng.random((b, n, m)) * 1e-3
    A[3] = -np.eye(n)                                             # one indefinite block: a non-zero info
    return A, B, C


def _block_cholesky(handle, ik, ok):
    n, m, b = 10, 5, 7
    A, B, C = _block_blocks(n, m, b)
    out = _outs(ok, M=((b, n + m, n + m), F8), info=(b, I4))
    return _call(handle, ops.block_cholesky, n, m, b, 0, _to(ik, A), _to(ik, B), _to(ik, C), **out)[1]


def _block_ldiv(handle, ik, ok):
    n, m, b, nrhs = 10, 5, 7, 3
    A, B, C = _block_blocks(n, m, b)
    A[3] = np.eye(n)
    M = np.zeros((b, n + m, n + m))
    ops.block_cholesky(handle, n, m, b, 0, A, B, C, M)
    rhs = np.random.default_rng(16).standard_normal((b, nrhs, n + m))
    return _call(handle, ops.block_ldiv, n, m, b, 0, _to(ik, M), nrhs, b=_to(ik, rhs))[1]   # b: in / out


def _sqp(handle, ik, ok):
    from oracle import sqp_dubins as S
    Z0, x0, xf, o = S.turn90_problem(7, N=11)
    out = _outs(ok, feas_p=(7, F8), feas_d=(7, F8), iters=(7, I4))
    out["Z"] = _to(ik, Z0)                                        # in / out: follows the inputs
    solves, out = _call(handle, ops.sqp_dubins, 7, o, _to(ik, x0), _to(ik, xf), **out)
    return dict(out, solves=np.array(solves))


def _kkt_factor_args(f):
    return [f[k] for k in ("Q", "R", "Hux", "A", "B", "D2", "C")]


def _kkt_factor(handle, ik, ok):
    """lqrb_kkt_factor_f64 in the given kinds; the kept factor is then used by a host-array solve."""
    f = _kkt_problem(n=5, m=2, N=8, b=9, mid_p=1)
    n, m, N, b, p, hm = f["n"], f["m"], f["N"], f["batch"], f["p"], f["hess_mode"]
    _, out = _call(handle, ops.kkt_factor, n, m, N, b, p, hm, 0, *[_to(ik, a) for a in _kkt_factor_args(f)],
                   **_outs(ok, info=(b, I4)))
    NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
    dz, mult = np.zeros((b, NN)), np.zeros((b, P))
    ops.kkt_solve_factored(handle, n, m, N, b, p, hm, False, 0, f["q"], f["r"], f["d"], f["c"], dz, mult)
    return dict(out, dz=dz, mult=mult)


def _kkt_solve_factored(handle, ik, ok):
    """A host-array factorisation, then lqrb_kkt_solve_factored_f64 in the given kinds."""
    f = _kkt_problem(n=5, m=2, N=8, b=9, mid_p=1)
    n, m, N, b, p, hm = f["n"], f["m"], f["N"], f["batch"], f["p"], f["hess_mode"]
    ops.kkt_factor(handle, n, m, N, b, p, hm, 0, *_kkt_factor_args(f))
    NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
    out = _outs(ok, dz=((b, NN), F8), mult=((b, P), F8), res=((b, NN), F8), info=(b, I4))
    args = [_to(ik, f[k]) for k in ("q", "r", "d", "c")]
    return _call(handle, ops.kkt_solve_factored, n, m, N, b, p, hm, False, 0, *args, **out)[1]


def _kkt_get_shur(handle, ik, ok):
    f = _kkt_problem(n=4, m=2, N=6, b=5, mid_p=1)
    n, m, N, b, p = f["n"], f["m"], f["N"], f["batch"], f["p"]
    P = _lib.num_cons(n, N, p)
    out = _outs(ok, S=((b, P, P), F8), hvec=((b, P), F8), U=((b, P, P), F8), info=(b, I4))
    return _call(handle, ops.kkt_get_shur, n, m, N, b, p, f["hess_mode"], 0, *[_to(ik, f[k]) for k in KKT_NAMES], **out)[1]


CASES = dict(riccati=_riccati, kkt_solve=_kkt_solve, kkt_residual=_kkt_residual, rollout=_rollout, lsq_solve=_lsq,
             block_cholesky=_block_cholesky, block_ldiv=_block_ldiv, sqp_dubins=_sqp, kkt_factor=_kkt_factor,
             kkt_solve_factored=_kkt_solve_factored, kkt_get_shur=_kkt_get_shur)


def _assert_equal(got, want):
    assert got.keys() == want.keys()
    for k in want:
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("entry", list(CASES))
def test_host_and_device_arrays_agree(handle, oracle_mod, entry):
    host = CASES[entry](handle, HOST, HOST)
    dev = CASES[entry](handle, DEV, DEV)
    _assert_equal(dev, host)
    if entry == "block_cholesky":
        assert host["info"][3] != 0


# ------------------------------------------------------------------ several host chunks on both copy streams
def _in_host_chunks(handle, run, **opts):
    """run() with host arrays in chunks of 32 instances (both copy streams) and with device arrays in one call;
    returns both results and the conditioning record of each."""
    for k, v in opts.items():
        handle.set_option(k, v)
    try:
        handle.set_option("host_chunk", 32)
        host = run(HOST)
        host_cond = handle.kkt_last_condition(70)
        handle.set_option("host_chunk", 0)
        dev = run(DEV)
        dev_cond = handle.kkt_last_condition(70)
    finally:
        handle.set_option("host_chunk", 0)
        handle.set_option("kkt_cond_bits", 6)
    return host, dev, host_cond, dev_cond


@pytest.mark.parametrize("n,m,kern", [(12, 4, "riccati_dmma<12,4>"), (7, 2, "padded")])
def test_riccati_in_host_chunks(handle, n, m, kern):
    host, dev, _, _ = _in_host_chunks(handle, lambda k: _riccati(handle, k, k, n=n, m=m, N=20, b=70))
    assert kern in handle.last_kernel, handle.last_kernel
    _assert_equal(host, dev)


@pytest.mark.parametrize("n,m,opts,kern", [(12, 4, {"kkt_cond_bits": 1}, "+kkt_coop["), (10, 3, {}, "padded")])
def test_kkt_solve_in_host_chunks(handle, n, m, opts, kern):
    f = _kkt_problem(n=n, m=m, N=10, b=70)
    host, dev, (bits_h, res_h), (bits_d, res_d) = _in_host_chunks(handle, lambda k: _kkt_solve(handle, k, k, f), **opts)
    assert kern in handle.last_kernel, handle.last_kernel
    _assert_equal(host, dev)
    assert (bits_d >= 0).all() and np.array_equal(bits_h, bits_d) and res_h == res_d
    if opts:
        assert res_d == int((bits_d >= 1).sum()) > 0


def test_kkt_residual_in_host_chunks(handle):
    f = _kkt_problem(n=5, m=2, N=12, b=70, mid_p=1)
    host, dev, _, _ = _in_host_chunks(handle, lambda k: _kkt_residual(handle, k, k, f))
    _assert_equal(host, dev)


# ------------------------------------------------------------------ host and device arrays in one call
@pytest.mark.parametrize("entry", ["riccati", "kkt_solve", "lsq_solve"])
def test_mixed_host_and_device_arrays(handle, entry):
    """Device arrays with a numpy `info`, and host inputs with device outputs: such a call is staged, and its results
    equal the all-device call."""
    want = CASES[entry](handle, DEV, DEV)
    _assert_equal(CASES[entry](handle, DEV, DEV_INFO_HOST), want)
    _assert_equal(CASES[entry](handle, HOST, DEV), want)
