"""lqrb_admm_cache_f64, lqrb_admm_solve_f64 and lqr_b200.mpc.BoxMPC on the GPU: the cache records and fixed-count solves
against oracle/admm.py (itself pinned to exact solutions in tests/test_oracle_admm.py) at shapes covering every group
width; converged solves against the refined dense KKT solve of the converged active set (multiplier signs included)
and, without bounds, against lqrb_riccati_f64 with the cached terminal cost; warm starts; failed instances inside a
batch; NULL references and bounds; host, device and chunked pointers; argument codes; the receding-horizon loop."""
import ctypes as C
import itertools

import numpy as np
import pytest

from lqr_b200 import _lib, ops, problems
from oracle import admm as oa
from oracle import dense_kkt
from tests.test_oracle_admm import _bounds, _kkt

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1), (3, 2), (4, 1), (6, 3), (8, 4), (12, 4), (16, 8), (24, 6), (32, 8)]
RHO = 1.0


def _setup(n, m, N, b, seed, unstable=False, state_bounds=True):
    """A batch of dare_lti_riccati draws with references, input bounds of 0.5 and (state_bounds) a box of 2 on the first
    state component from knot 6 on: both bind on a good share of knots for x0 ~ 3 N(0, 1)."""
    p = problems.dare_lti_riccati(n, m, N, b, seed=seed, unstable=unstable)
    rng = np.random.default_rng(seed + 1)
    a = dict(x0=3.0 * p["x0"], xref=0.5 * rng.standard_normal((b, N, n)), uref=0.2 * rng.standard_normal((b, N - 1, m)),
             umin=np.full((b, N - 1, m), -0.5), umax=np.full((b, N - 1, m), 0.5))
    if state_bounds:
        a["xmin"], a["xmax"] = np.full((b, N - 1, n), -np.inf), np.full((b, N - 1, n), np.inf)
        a["xmin"][:, 4:, 0], a["xmax"][:, 4:, 0] = -2.0, 2.0
    return p, a


def _rec(cache, n, m, i):
    """instance i of GPU cache records as the oracle's cache dict"""
    s = ops.admm_cache_split(cache, n, m)
    return {k: (float(v[i]) if k == "rho" else v[i]) for k, v in s.items()}


def _oracle(cache, n, m, N, a, i, **kw):
    get = lambda k: None if a.get(k) is None else a[k][i]  # noqa: E731
    return oa.solve(_rec(cache, n, m, i), a["x0"][i], N, get("xref"), get("uref"), get("umin"), get("umax"),
                    get("xmin"), get("xmax"), **kw)


def _rel(a, b):
    return np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300)


@pytest.mark.parametrize("n,m", SHAPES)
def test_cache_matches_oracle(handle, n, m):
    b = 5
    p, _ = _setup(n, m, 2, b, seed=n + m, unstable=n % 2 == 0)
    cache, info = ops.admm_cache_problem(p, RHO, handle=handle)
    assert (info == 0).all(), info
    for i in range(b):
        o = oa.cache(p["A"][i], p["B"][i], p["Q"][i], p["R"][i], RHO)
        g = _rec(cache, n, m, i)
        for k in ("A", "B", "Q", "R"):
            assert np.array_equal(g[k], o[k]), k
        assert g["rho"] == RHO
        tol = 1e-10 if n <= 16 else 1e-9
        for k in ("K", "C1", "C2", "Qf"):
            assert _rel(g[k], o[k]) <= tol, (i, k, _rel(g[k], o[k]))


@pytest.mark.parametrize("n,m", SHAPES)
def test_fixed_count_solve_matches_oracle(handle, n, m):
    b, N, its = 6, 12, 25
    p, a = _setup(n, m, N, b, seed=2 * n + m, unstable=n % 2 == 1)
    cache, info = ops.admm_cache_problem(p, RHO, handle=handle)
    assert (info == 0).all()
    X, U, iters, res, sinfo = ops.admm_solve_problem(cache, a["x0"], N, a["xref"], a["uref"], a["umin"], a["umax"],
                                                     a["xmin"], a["xmax"], max_iter=its, eps_pri=0.0, eps_dual=0.0,
                                                     handle=handle)
    assert handle.last_kernel.startswith(f"admm<G={max(4, 1 << (n - 1).bit_length())}>"), handle.last_kernel
    assert (sinfo == 1).all() and (iters == its).all(), (sinfo, iters)
    for i in range(b):
        r = _oracle(cache, n, m, N, a, i, max_iter=its)
        scale = max(np.abs(r["X"]).max(), np.abs(r["U"]).max())
        assert np.abs(X[i] - r["X"]).max() <= 1e-10 * scale and np.abs(U[i] - r["U"]).max() <= 1e-10 * scale, i
        assert abs(res[i, 0] - r["r_pri"]) <= 1e-10 * scale and abs(res[i, 1] - r["r_dual"]) <= 1e-10 * scale


def _cartpole(b, N):
    """the reference's cartpole linearisation (last knot of its fixture), one draw of x0 per instance"""
    f = problems.cartpole_fixture(101)
    rng = np.random.default_rng(7)
    p = dict(A=np.repeat(f["A"][0, -1][None], b, 0), B=np.repeat(f["B"][0, -1][None], b, 0),
             Q=np.repeat(np.eye(4)[None], b, 0), R=np.repeat(0.1 * np.eye(1)[None], b, 0))
    return p, dict(x0=rng.standard_normal((b, 4)), xref=np.zeros((b, N, 4)), uref=np.zeros((b, N - 1, 1)))


@pytest.mark.parametrize("case", ["cartpole", "4-1-unstable", "12-4-stable", "12-4-unstable"])
def test_converged_solve_satisfies_the_kkt_conditions(handle, case):
    """bounds from each instance's unconstrained solution, as in tests/test_oracle_admm.py, so that they bind and the
    problem stays feasible"""
    N, b = 50, 4
    if case == "cartpole":
        p, a = _cartpole(b, N)
        n, m = 4, 1
    else:
        n, m, st = case.split("-")
        n, m = int(n), int(m)
        p, a = _setup(n, m, N, b, seed=n + 4, unstable=st == "unstable", state_bounds=False)
    # the cartpole with a cart-position box takes 1e4-1e5 iterations: input bounds only there
    sb = case != "cartpole"
    bs = [_bounds(oa.cache(p["A"][i], p["B"][i], p["Q"][i], p["R"][i], RHO), a["x0"][i], a["xref"][i], a["uref"][i],
                  sb, N=N) for i in range(b)]
    for k in ("umin", "umax", "xmin", "xmax"):
        a[k] = np.stack([x[k] for x in bs]) if sb or k[0] == "u" else np.full((b, N - 1, n), np.inf if k == "xmax" else -np.inf)
    cache, info = ops.admm_cache_problem(p, RHO, handle=handle)
    assert (info == 0).all()
    eps = 1e-10
    state = np.zeros((b, 2 * (N - 1) * (n + m)))
    X, U, iters, res, sinfo = ops.admm_solve_problem(cache, a["x0"], N, a["xref"], a["uref"], a["umin"], a["umax"],
                                                     a["xmin"], a["xmax"], state=state, max_iter=50000, eps_pri=eps,
                                                     eps_dual=eps, handle=handle)
    assert (sinfo == 0).all(), (sinfo, iters)
    assert (res[:, 0] <= eps).all() and (res[:, 1] <= eps).all()
    Km, Kn = (N - 1) * m, (N - 1) * n
    w, active_x, active_u = n + m, 0, 0
    for i in range(b):
        z, y = state[i, :Km].reshape(N - 1, m), state[i, Km:2 * Km].reshape(N - 1, m)
        v, g = state[i, 2 * Km:2 * Km + Kn].reshape(N - 1, n), state[i, 2 * Km + Kn:].reshape(N - 1, n)
        rows, mult = [], []
        for k in range(N - 1):
            for j in range(m):
                if z[k, j] in (a["umin"][i, k, j], a["umax"][i, k, j]):
                    rows.append((k * w + n + j, z[k, j]))
                    mult.append(RHO * y[k, j])
            for j in range(n):
                if v[k, j] in (a["xmin"][i, k, j], a["xmax"][i, k, j]):
                    rows.append(((k + 1) * w + j, v[k, j]))
                    mult.append(RHO * g[k, j])
        active_u += sum(col % w >= n for col, _ in rows)
        active_x += sum(col % w < n for col, _ in rows)
        xr = np.zeros((N, n)) if a["xref"] is None else a["xref"][i]
        ur = np.zeros((N - 1, m)) if a["uref"] is None else a["uref"][i]
        dz, lam = dense_kkt.solve_refined(*_kkt(_rec(cache, n, m, i), a["x0"][i], xr, ur, rows, N=N))
        scale = max(1.0, np.abs(dz).max())
        assert np.abs(oa.primals(X[i], U[i]) - dz).max() <= 1e-6 * scale, i
        lscale = max(1.0, np.abs(lam).max())
        if rows:
            assert np.abs(lam[n + Kn:] - np.array(mult)).max() <= 1e-6 * lscale, i
        tol = 1e-6 * lscale
        assert np.all(y[z == a["umax"][i]] >= -tol) and np.all(y[z == a["umin"][i]] <= tol)
        assert np.all(g[v == a["xmax"][i]] >= -tol) and np.all(g[v == a["xmin"][i]] <= tol)
        free_u = (z > a["umin"][i]) & (z < a["umax"][i])
        free_x = (v > a["xmin"][i]) & (v < a["xmax"][i])
        assert np.abs(y[free_u]).max(initial=0.0) <= tol and np.abs(g[free_x]).max(initial=0.0) <= tol
    assert active_u > 0 and (active_x > 0 or not sb), (active_u, active_x)


@pytest.mark.parametrize("n,m,unstable", [(4, 1, False), (6, 3, True), (12, 4, True)])
def test_unbounded_solve_equals_riccati_with_the_cached_terminal_cost(handle, n, m, unstable):
    N, b = 40, 4
    p, a = _setup(n, m, N, b, seed=n * m, unstable=unstable, state_bounds=False)
    cache, info = ops.admm_cache_problem(p, RHO, handle=handle)
    X, U, iters, _, sinfo = ops.admm_solve_problem(cache, a["x0"], N, a["xref"], a["uref"], max_iter=20000,
                                                   eps_pri=1e-13, eps_dual=1e-13, handle=handle)
    assert (info == 0).all() and (sinfo == 0).all(), (sinfo, iters)
    Qf = ops.admm_cache_split(cache, n, m)["Qf"]
    rep = lambda M: np.repeat(M[:, None], N - 1, axis=1)  # noqa: E731
    prob = dict(n=n, m=m, N=N, lti=False, A=rep(p["A"]), B=rep(p["B"]), Q=rep(p["Q"]), R=rep(p["R"]),
                q=-np.einsum("bij,bkj->bki", p["Q"], a["xref"][:, :-1]), r=-np.einsum("bij,bkj->bki", p["R"], a["uref"]),
                Qf=np.ascontiguousarray(Qf), qf=-np.einsum("bij,bj->bi", Qf, a["xref"][:, -1]), x0=a["x0"])
    Xr, Ur, _, _, rinfo = ops.riccati_solve_problem(prob, want_gains=False, handle=handle)
    assert (rinfo == 0).all()
    for i in range(b):
        scale = max(np.abs(Xr[i]).max(), np.abs(Ur[i]).max())
        assert np.abs(X[i] - Xr[i]).max() <= 1e-9 * scale and np.abs(U[i] - Ur[i]).max() <= 1e-9 * scale, i


@pytest.mark.parametrize("n,m", [(4, 1), (12, 4), (32, 8)])
def test_warm_start_continues_the_cold_iteration_bitwise(handle, n, m):
    N, b = 20, 9
    p, a = _setup(n, m, N, b, seed=n + 11, unstable=True)
    cache, _ = ops.admm_cache_problem(p, RHO, handle=handle)
    args = [a[k] for k in ("xref", "uref", "umin", "umax", "xmin", "xmax")]
    L = 2 * (N - 1) * (n + m)
    s1, s2 = np.zeros((b, L)), np.zeros((b, L))
    ops.admm_solve_problem(cache, a["x0"], N, *args, state=s1, max_iter=6, eps_pri=0, eps_dual=0, handle=handle)
    Xw, Uw, itw, resw, _ = ops.admm_solve_problem(cache, a["x0"], N, *args, state=s1, warm=True, max_iter=5, eps_pri=0,
                                                  eps_dual=0, handle=handle)
    Xc, Uc, itc, resc, _ = ops.admm_solve_problem(cache, a["x0"], N, *args, state=s2, max_iter=11, eps_pri=0, eps_dual=0,
                                                  handle=handle)
    assert np.array_equal(Xw, Xc) and np.array_equal(Uw, Uc) and np.array_equal(resw, resc)
    assert np.array_equal(s1, s2) and (itw == 5).all() and (itc == 11).all()


def _bad_batch(n, m, N):
    p, a = _setup(n, m, N, 9, seed=5, unstable=True)
    ins = lambda x: np.insert(x, [2, 4, 6], x[:3], axis=0)  # noqa: E731
    p2 = {k: ins(p[k]) for k in "ABQR"}
    a2 = {k: ins(v) for k, v in a.items()}
    p2["A"][2], p2["B"][2] = 1.5 * np.eye(n), 0.0  # no stabilising DARE solution: a NaN cache record
    a2["x0"][5, 0] = np.nan                        # NaN input
    a2["umin"][8, 3, 0] = 1.0                      # empty box: umin > umax = 0.5
    return p, a, p2, a2, np.setdiff1d(np.arange(12), [2, 5, 8])


@pytest.mark.parametrize("n,m", [(4, 1), (12, 4)])
def test_failed_instances_leave_the_batch_alone(handle, n, m):
    N = 15
    p, a, p2, a2, good = _bad_batch(n, m, N)
    c0, ci0 = ops.admm_cache_problem(p, RHO, handle=handle)
    c1, ci1 = ops.admm_cache_problem(p2, RHO, handle=handle)
    assert (ci0 == 0).all() and ci1[2] == 1 and (ci1[good] == 0).all() and (ci1[[5, 8]] == 0).all(), ci1
    assert np.isnan(c1[2]).all() and np.array_equal(c1[good], c0)
    keys = ("xref", "uref", "umin", "umax", "xmin", "xmax")
    L = 2 * (N - 1) * (n + m)
    s0, s1 = np.zeros((9, L)), np.zeros((12, L))
    r0 = ops.admm_solve_problem(c0, a["x0"], N, *(a[k] for k in keys), state=s0, max_iter=500, eps_pri=1e-8,
                                eps_dual=1e-8, handle=handle)
    r1 = ops.admm_solve_problem(c1, a2["x0"], N, *(a2[k] for k in keys), state=s1, max_iter=500, eps_pri=1e-8,
                                eps_dual=1e-8, handle=handle)
    info = r1[4]
    assert info[2] == 2 and info[5] == 2 and info[8] == 3, info
    for x0, x1 in zip(r0, r1):
        assert np.array_equal(x1[good], x0)
    assert np.array_equal(s1[good], s0)
    for x in (r1[0], r1[1], r1[3], s1):
        assert np.isnan(x[[2, 5, 8]]).all()


def test_null_references_and_bounds_match_the_oracle(handle):
    n, m, N, b, its = 6, 3, 10, 3, 8
    p, a = _setup(n, m, N, b, seed=21, unstable=True)
    a["umax"][:, 2] = np.inf   # infinite entries are legal
    a["xmin"][:, 5, 1] = -np.inf
    cache, _ = ops.admm_cache_problem(p, RHO, handle=handle)
    keys = ("xref", "uref", "umin", "umax", "xmin", "xmax")
    for mask in itertools.product([False, True], repeat=len(keys)):
        sub = dict(x0=a["x0"], **{k: (a[k] if on else None) for k, on in zip(keys, mask)})
        X, U, _, _, info = ops.admm_solve_problem(cache, a["x0"], N, *(sub[k] for k in keys), max_iter=its, eps_pri=0,
                                                  eps_dual=0, handle=handle)
        assert (info == 1).all(), (mask, info)
        for i in range(b):
            r = _oracle(cache, n, m, N, sub, i, max_iter=its)
            scale = max(np.abs(r["X"]).max(), np.abs(r["U"]).max())
            assert np.abs(X[i] - r["X"]).max() <= 1e-10 * scale and np.abs(U[i] - r["U"]).max() <= 1e-10 * scale, mask


@pytest.mark.parametrize("n,m", [(4, 1), (24, 6)])
def test_host_device_chunked_and_repeated_runs_are_bitwise_equal(handle, n, m):
    import torch
    N, b = 16, 37
    p, a = _setup(n, m, N, b, seed=3, unstable=True)
    keys = ("xref", "uref", "umin", "umax", "xmin", "xmax")
    L = 2 * (N - 1) * (n + m)
    cache, cinfo = ops.admm_cache_problem(p, RHO, handle=handle)

    def run(c, **kw):
        s = np.zeros((b, L))
        out = ops.admm_solve_problem(c, a["x0"], N, *(a[k] for k in keys), state=s, max_iter=300, eps_pri=1e-7,
                                     eps_dual=1e-7, handle=handle, **kw)
        return out + (s,)
    ref = run(cache)
    handle.set_option("host_chunk", 8)
    try:
        cache_c, cinfo_c = ops.admm_cache_problem(p, RHO, handle=handle)
        chunked = run(cache)
    finally:
        handle.set_option("host_chunk", 0)
    again = run(cache)
    assert np.array_equal(cache_c, cache) and np.array_equal(cinfo_c, cinfo)
    for x, y, z in zip(ref, chunked, again):
        assert np.array_equal(x, y) and np.array_equal(x, z)
    # device-resident: torch tensors in the ABI's layouts
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    cmd = lambda x: dev(np.swapaxes(x, -1, -2))  # noqa: E731
    cd = torch.empty(b, ops.admm_cache_doubles(n, m), dtype=torch.float64, device="cuda")
    ops.admm_cache(handle, n, m, b, RHO, cmd(p["A"]), cmd(p["B"]), cmd(p["Q"]), cmd(p["R"]), cd)
    Z = torch.empty(b, _lib.num_vars(n, m, N), dtype=torch.float64, device="cuda")
    st = torch.empty(b, L, dtype=torch.float64, device="cuda")
    it, info = (torch.empty(b, dtype=torch.int32, device="cuda") for _ in range(2))
    res = torch.empty(b, 2, dtype=torch.float64, device="cuda")
    ops.admm_solve(handle, n, m, N, b, cd, dev(a["x0"]), Z, *(dev(a[k]) for k in keys), state=st, max_iter=300,
                   eps_pri=1e-7, eps_dual=1e-7, iters=it, res=res, info=info)
    handle.synchronize()
    assert np.array_equal(cd.cpu().numpy(), cache)
    Xd, Ud = ops.split_primals(Z.cpu().numpy(), n, m, N)
    assert np.array_equal(Xd, ref[0]) and np.array_equal(Ud, ref[1]) and np.array_equal(it.cpu().numpy(), ref[2])
    assert np.array_equal(res.cpu().numpy(), ref[3]) and np.array_equal(info.cpu().numpy(), ref[4])
    assert np.array_equal(st.cpu().numpy(), ref[5])


def test_argument_codes(handle):
    L, h = _lib.lib(), handle._h
    a = np.zeros(1 << 16)
    p = a.ctypes.data
    i32 = np.zeros(64, dtype=np.int32)

    def cache(n=4, m=2, b=2, rho=1.0, A=1, B=1, Q=1, R=1, c=1):
        s = lambda f: p if f else None  # noqa: E731
        return L.lqrb_admm_cache_f64(h, n, m, b, rho, s(A), s(B), s(Q), s(R), s(c), None)

    assert cache(n=0) == -2 and cache(n=33) == -2 and cache(m=0) == -3 and cache(m=5) == -3 and cache(b=-1) == -4
    assert cache(rho=0.0) == -5 and cache(rho=-1.0) == -5 and cache(rho=np.inf) == -5 and cache(rho=np.nan) == -5
    assert cache(A=0) == -6 and cache(B=0) == -7 and cache(Q=0) == -8 and cache(R=0) == -9 and cache(c=0) == -10
    assert cache(b=0) == 0
    assert L.lqrb_admm_cache_f64(None, 4, 2, 2, 1.0, p, p, p, p, p, None) == -1

    def solve(n=4, m=2, N=10, b=2, flags=0, it=10, ep=0.0, ed=0.0, opts=True, c=1, x0=1, state=0, Z=1):
        o = _lib.AdmmOptions(max_iter=it, eps_pri=ep, eps_dual=ed)
        s = lambda f: p if f else None  # noqa: E731
        return L.lqrb_admm_solve_f64(h, n, m, N, b, flags, C.byref(o) if opts else None, s(c), s(x0), None, None,
                                     None, None, None, None, s(state), s(Z), None, None, i32.ctypes.data)

    assert solve(n=0) == -2 and solve(n=33) == -2 and solve(m=0) == -3 and solve(m=5) == -3 and solve(N=1) == -4
    assert solve(b=-1) == -5 and solve(flags=1) == -6 and solve(flags=_lib.FLAG_WARM_START) == -6
    assert solve(opts=False) == -7 and solve(it=0) == -7 and solve(ep=-1.0) == -7 and solve(ed=np.nan) == -7
    assert solve(c=0) == -8 and solve(x0=0) == -9 and solve(Z=0) == -17 and solve(b=0) == 0
    # the admission limit: one instance's working set (2n^2 + 2nm + m^2 + (N-1)(6n + 6m) doubles) over 227 KB
    assert solve(n=32, m=8, N=111, b=0) == 0 and solve(n=32, m=8, N=112, b=0) == -4
    assert "227 KB" in _lib.lib().lqrb_last_error_string(h).decode()
    assert L.lqrb_admm_solve_f64(None, 4, 2, 10, 2, 0, None, p, p, None, None, None, None, None, None, None, p, None,
                                 None, None) == -1


def test_box_mpc_receding_horizon_matches_ops(handle):
    import torch
    from lqr_b200.mpc import BoxMPC
    n, m, N, b, steps = 4, 1, 30, 8, 5
    p, a = _cartpole(b, N)
    a.update(umin=np.full((b, N - 1, m), -1.0), umax=np.full((b, N - 1, m), 1.0),
             xmin=np.full((b, N - 1, n), -np.inf), xmax=np.full((b, N - 1, n), np.inf))
    a["xmin"][:, 9:, 0], a["xmax"][:, 9:, 0] = -0.5, 0.5
    t = lambda x: torch.tensor(x, dtype=torch.float64, device="cuda")  # noqa: E731
    mpc = BoxMPC(t(p["A"][:1]), t(p["B"][:1]), t(p["Q"][:1]), t(p["R"][:1]), RHO)  # broadcast over the batch of x0
    with pytest.raises(TypeError):
        BoxMPC(*(torch.tensor(p[k]) for k in "ABQR"), RHO)
    cache, _ = ops.admm_cache_problem({k: p[k] for k in "ABQR"}, RHO, handle=handle)
    state = np.zeros((b, 2 * (N - 1) * (n + m)))
    x, xs = a["x0"].copy(), t(a["x0"])
    for k in range(steps):
        X, U, info = mpc.solve(xs, umin=-1.0, umax=1.0, xmin=t(a["xmin"][:1]), xmax=t(a["xmax"][:1]), max_iter=200,
                               eps=1e-7)
        Xo, Uo, _, _, io = ops.admm_solve_problem(cache, x, N, None, None, a["umin"], a["umax"], a["xmin"], a["xmax"],
                                                  state=state, warm=k > 0, max_iter=200, eps_pri=1e-7, eps_dual=1e-7,
                                                  handle=handle)
        assert np.array_equal(X.cpu().numpy(), Xo) and np.array_equal(U.cpu().numpy(), Uo)
        assert np.array_equal(info.cpu().numpy(), io)
        assert np.array_equal(mpc.state.cpu().numpy(), state) and np.array_equal(mpc.cache.cpu().numpy(), cache)
        # apply the first control and move on
        x = x @ p["A"][0].T + Uo[:, 0] @ p["B"][0].T
        xs = t(x)
