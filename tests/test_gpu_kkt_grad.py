"""lqrb_kkt_grad_f64 and lqr_b200.autograd.kkt_solve on the GPU: gradients of l(dz, mult) through the constrained KKT
solve against the CPU gradient oracle (oracle/kkt_grad.py: the adjoint formulas on the refined dense solve, itself
pinned against finite differences in tests/test_oracle_kkt_grad.py) on one shape of every kernel family that solves
the adjoint problem; the Riccati gradient on the same problem written as a KKT system; finite differences through the
library's own forward solve; host vs device pointers; argument errors; the handle state the call must leave alone;
determinism; torch gradcheck."""

import numpy as np
import pytest

from lqr_b200 import _lib, ops, problems

pytestmark = pytest.mark.gpu

NAMES = ("Q", "R", "Hux", "q", "r", "A", "B", "d", "D2", "C", "c")


@pytest.fixture
def option(handle):
    """sets handle options for one test and restores their defaults"""
    set_ = {}

    def setter(name, value, default):
        set_[name] = default
        handle.set_option(name, value)
    yield setter
    for name, default in set_.items():
        handle.set_option(name, default)


def _ragged(prob, seed, hi):
    """a random number (0..hi) of the stage rows on every interior knot"""
    rng = np.random.default_rng(seed)
    p = prob["p"].copy()
    for k in range(1, prob["N"] - 1):
        p[k] = int(rng.integers(0, hi + 1))
        prob["C"][k] = prob["C"][k][:, :p[k]]
        prob["c"][k] = prob["c"][k][:, :p[k]]
    prob["p"] = p
    return prob


def _free_final(prob):
    prob["p"] = prob["p"].copy()
    prob["p"][-1] = 0
    b = prob["q"].shape[0]
    prob["C"][-1] = np.zeros((b, 0, prob["n"]))
    prob["c"][-1] = np.zeros((b, 0))
    return prob


def _solve_and_grad(handle, prob, seed=0):
    dz, mult, info = ops.kkt_solve_problem(prob, handle=handle)
    assert (info == 0).all(), handle.last_kernel
    solve_kernel = handle.last_kernel
    rng = np.random.default_rng(seed)
    dzb, mb = rng.standard_normal(dz.shape), rng.standard_normal(mult.shape)
    g, ginfo = ops.kkt_grad_problem(prob, dz, mult, dzb, mb, handle=handle)
    assert (ginfo == 0).all()
    assert handle.last_kernel == solve_kernel + " + kkt_grad", (handle.last_kernel, solve_kernel)
    return dz, mult, dzb, mb, g


def _flat(v):
    if v is None:
        return np.zeros(0)
    if isinstance(v, list):
        return np.concatenate([x.reshape(-1) for x in v]) if v else np.zeros(0)
    return v.reshape(-1)


def _rel_errors(prob, dzb, mb, g):
    from oracle.kkt_grad import kkt_grad
    go = kkt_grad(prob, dzb, mb)
    out = {}
    for k in NAMES:
        a, b = _flat(g[k]), _flat(go[k])
        assert a.shape == b.shape, k
        if b.size:
            out[k] = np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)
    return out


def _check_against_oracle(prob, dzb, mb, g, tol=1e-9):
    for k, err in _rel_errors(prob, dzb, mb, g).items():
        assert err <= tol, (k, err)


# (n, m, N, batch, generator options, kernel the forward and adjoint solves run on)
FAMILIES = {
    "tpi-dubins": (3, 2, 41, 3, dict(dubins=True), "kkt_tpi<3,2"),
    "tpi-free-final": (3, 2, 20, 3, dict(free=True), "kkt_tpi<3,2,p=3/0/0"),
    "hw": (12, 4, 20, 3, dict(), "kkt_hw<12,4"),
    "wp-dense": (8, 2, 16, 3, dict(hess=0), "kkt_wp_dmma<8,2"),
    "wp-per-knot-rows": (8, 2, 20, 3, dict(mid_p=1, ragged=True), "kkt_wp_dmma<8,2,p=8/per-knot<=1/8"),
    "cta-stage-rows": (16, 8, 10, 3, dict(mid_p=2), "kkt_cta_dmma<16,8,p=16/2/16"),
    "padded-10-3": (10, 3, 16, 3, dict(mid_p=1), "kkt_wp_dmma<12,4"),
    "padded-24-6": (24, 6, 8, 3, dict(), "kkt_cta_dmma<24,8"),
    "coop-explicit-D2": (3, 2, 8, 3, dict(d2x=True, hess=0, mid_p=1), "kkt_coop"),
}


def _family_problem(n, m, N, b, o, seed):
    if o.get("dubins"):
        return problems.dubins_kkt_batch(b, seed=seed, N=N, mid_p=1)
    prob = problems.random_lqr_kkt(n, m, N, b, seed=seed, mid_p=o.get("mid_p", 0), hess_mode=o.get("hess", 1),
                                   explicit_D2=o.get("d2x", False))
    if o.get("ragged"):
        prob = _ragged(prob, seed, o["mid_p"])
        assert len(set(prob["p"][1:-1].tolist())) > 1
    if o.get("free"):
        prob = _free_final(prob)
    return prob


@pytest.mark.parametrize("family", list(FAMILIES))
def test_gradients_match_oracle_on_every_family(handle, family):
    n, m, N, b, o, kern = FAMILIES[family]
    prob = _family_problem(n, m, N, b, o, seed=3 * n + m)
    _, _, dzb, mb, g = _solve_and_grad(handle, prob, seed=n)
    assert handle.last_kernel.startswith(kern), handle.last_kernel
    assert ("padded" in handle.last_kernel) == family.startswith("padded"), handle.last_kernel
    _check_against_oracle(prob, dzb, mb, g)


def test_gradients_on_the_cooperative_kernel_variant(handle, option):
    option("kkt_variant", 2, 0)
    prob = problems.random_lqr_kkt(12, 4, 12, 3, seed=5, mid_p=2, hess_mode=2)
    _, _, dzb, mb, g = _solve_and_grad(handle, prob, seed=5)
    assert handle.last_kernel.startswith("kkt_coop")
    _check_against_oracle(prob, dzb, mb, g)


def test_gradients_through_the_re_solve_of_ill_conditioned_instances(handle, option):
    """kkt_cond_bits = 0 flags every instance of the tuned kernel, so the adjoint problem is solved again by the
    Cholesky-based kernel, as the forward one is."""
    option("kkt_cond_bits", 0, 6)
    prob = problems.random_lqr_kkt(12, 4, 14, 3, seed=6, mid_p=1)
    dz, mult, info = ops.kkt_solve_problem(prob, handle=handle)
    assert "kkt_coop[3 ill-conditioned]" in handle.last_kernel, handle.last_kernel
    rng = np.random.default_rng(6)
    dzb, mb = rng.standard_normal(dz.shape), rng.standard_normal(mult.shape)
    g, ginfo = ops.kkt_grad_problem(prob, dz, mult, dzb, mb, handle=handle)
    assert (ginfo == 0).all() and handle.last_kernel.endswith("kkt_coop[3 ill-conditioned] + kkt_grad")
    _check_against_oracle(prob, dzb, mb, g)


@pytest.mark.parametrize("n,m", [(4, 1), (12, 4)])
def test_riccati_problem_as_kkt_reproduces_the_riccati_gradient(handle, n, m):
    """dense_kkt.riccati_as_kkt writes an LQR as a KKT system with initial-condition rows c_1 = -x0: lqrb_kkt_grad_f64
    must give lqrb_riccati_grad_f64's gA, gB, gR, gr; gQ_k, gq_k for k < N-1 and gQf, gqf at knot N-1; gx0 = -gc_1."""
    from oracle import dense_kkt
    N, b = 15, 3
    prob = problems.random_lqr_riccati(n, m, N, b, seed=n, dt=0.05)
    kp = dense_kkt.riccati_as_kkt(prob)
    dz, mult, info = ops.kkt_solve_problem(kp, handle=handle)
    assert (info == 0).all()
    dZ = np.random.default_rng(1).standard_normal(dz.shape)
    gk, _ = ops.kkt_grad_problem(kp, dz, mult, dZ, None, handle=handle)
    X, U, _, _, _ = ops.riccati_solve_problem(prob, want_gains=False, handle=handle)
    Z = np.concatenate([np.concatenate([X[:, :-1], U], axis=2).reshape(b, -1), X[:, -1]], axis=1)
    gr_, _ = ops.riccati_grad_problem(prob, Z, dZ, handle=handle)

    def close(a, b_):
        assert np.linalg.norm(a - b_) <= 1e-9 * np.linalg.norm(b_)
    for k in ("A", "B", "R", "r"):
        close(gk[k], gr_[k])
    close(gk["Q"][:, :N - 1], gr_["Q"])
    close(gk["q"][:, :N - 1], gr_["q"])
    close(gk["Q"][:, N - 1], gr_["Qf"])
    close(gk["q"][:, N - 1], gr_["qf"])
    close(-gk["c"][0], gr_["x0"])


def _direction(prob, rng):
    D = {}
    for k in NAMES:
        v = prob.get(k)
        if v is None:
            D[k] = None
        elif isinstance(v, list):
            D[k] = [rng.standard_normal(np.shape(x)) for x in v]
        else:
            D[k] = rng.standard_normal(np.shape(v))
    for k in ("Q", "R"):
        D[k] = D[k] + np.swapaxes(D[k], -1, -2)
    return D


def _step(prob, D, s):
    p = dict(prob)
    for k, v in D.items():
        if v is None:
            continue
        p[k] = [x + s * dx for x, dx in zip(prob[k], v)] if isinstance(v, list) else prob[k] + s * v
    return p


@pytest.mark.parametrize("n,m,mid_p,hess,d2x", [(12, 4, 2, 1, False), (6, 3, 1, 0, True), (16, 8, 1, 2, False)])
def test_directional_finite_difference_through_the_library(handle, n, m, mid_p, hess, d2x):
    """sum(g * D) against (l(p + hD) - l(p - hD)) / 2h, l = sum(dz_bar * dz) + sum(mult_bar * mult) solved by the library
    itself"""
    b = 2
    prob = problems.random_lqr_kkt(n, m, 10, b, seed=9, mid_p=mid_p, hess_mode=hess, explicit_D2=d2x)
    _, _, dzb, mb, g = _solve_and_grad(handle, prob, seed=1)
    D = _direction(prob, np.random.default_rng(2))
    h = 1e-6

    def loss(s):
        dz, mult, _ = ops.kkt_solve_problem(_step(prob, D, s * h), handle=handle)
        return (dz * dzb).sum(axis=1) + (mult * mb).sum(axis=1)
    fd = (loss(1) - loss(-1)) / (2 * h)
    an = np.zeros(b)
    for k in NAMES:
        if D[k] is None:
            continue
        pairs = zip(g[k], D[k]) if isinstance(D[k], list) else [(g[k], D[k])]
        for gk, dk in pairs:
            an += (gk * dk).reshape(b, -1).sum(axis=1)
    np.testing.assert_allclose(an, fd, rtol=1e-6)


def _abi_args(prob):
    f = ops.kkt_flatten(prob)
    return f, [f[k] for k in ("Q", "R", "Hux", "A", "B", "D2", "C")]


def _abi_grads(f, dense=False, d2x=False):
    n, m, N, b = f["n"], f["m"], f["N"], f["batch"]
    return [np.zeros_like(f["Q"]), np.zeros_like(f["R"]), np.zeros((b, N - 1, n, m)) if dense else None,
            np.zeros_like(f["q"]), np.zeros_like(f["r"]), np.zeros_like(f["A"]), np.zeros_like(f["B"]),
            np.zeros_like(f["d"]), np.zeros_like(f["D2"]) if d2x else None, np.zeros_like(f["C"]), np.zeros_like(f["c"])]


def test_host_and_device_pointers_agree_bitwise_over_uneven_chunks(handle, option):
    import torch
    prob = problems.random_lqr_kkt(6, 3, 20, 100, seed=7, mid_p=1, hess_mode=0, explicit_D2=False)
    dz, mult, dzb, mb, g = _solve_and_grad(handle, prob, seed=7)  # host, default chunking
    f, ins = _abi_args(prob)
    n, m, N, b = 6, 3, 20, 100
    option("host_chunk", 32, 0)  # 32 + 32 + 32 + 4 instances
    outs_h = _abi_grads(f, dense=True)
    info_h = np.zeros(b, dtype=np.int32)
    ops.kkt_grad(handle, n, m, N, b, f["p"], 0, 0, *ins, dz, mult, dzb, mb, *outs_h, info_h)
    cuda = [None if a is None else torch.from_numpy(a).cuda() for a in ins + [dz, mult, dzb, mb]]
    outs_d = [None if a is None else torch.zeros(a.shape, dtype=torch.float64, device="cuda") for a in outs_h]
    info_d = torch.zeros(b, dtype=torch.int32, device="cuda")
    handle.set_stream(torch.cuda.current_stream().cuda_stream or 1)  # 1 = cudaStreamLegacy (torch's default stream)
    ops.kkt_grad(handle, n, m, N, b, f["p"], 0, 0, *cuda, *outs_d, info_d)
    torch.cuda.synchronize()
    handle.set_stream(None)
    for a, d in zip(outs_h, outs_d):
        if a is not None:
            assert np.array_equal(a, d.cpu().numpy())
    assert np.array_equal(np.swapaxes(outs_h[0], -1, -2), g["Q"]) and np.array_equal(outs_h[10], np.concatenate(g["c"], 1))


def test_null_outputs_null_cotangents_and_batch_zero(handle):
    prob = problems.random_lqr_kkt(4, 2, 9, 5, seed=1, mid_p=1)
    dz, mult, dzb, mb, g = _solve_and_grad(handle, prob, seed=2)
    f, ins = _abi_args(prob)
    n, m, N, b, p = 4, 2, 9, 5, f["p"]
    gA, gc = np.zeros_like(f["A"]), np.zeros_like(f["c"])
    ops.kkt_grad(handle, n, m, N, b, p, 1, 0, *ins, dz, mult, dzb, mb, gA=gA, gc=gc)
    assert np.array_equal(np.swapaxes(gA, -1, -2), g["A"]) and np.array_equal(gc, np.concatenate(g["c"], 1))
    ops.kkt_grad(handle, n, m, N, 0, p, 1, 0, *ins, dz, mult, dzb, mb, gA=gA)  # batch 0: nothing to do
    # a NULL cotangent reads as zeros
    for zb, mbb in ((dzb, None), (None, mb)):
        g1, _ = ops.kkt_grad_problem(prob, dz, mult, zb, mbb, handle=handle)
        g0, _ = ops.kkt_grad_problem(prob, dz, mult, np.zeros_like(dzb) if zb is None else zb,
                                     np.zeros_like(mb) if mbb is None else mbb, handle=handle)
        for k in NAMES:
            assert np.array_equal(_flat(g1[k]), _flat(g0[k])), k


def test_argument_codes(handle):
    prob = problems.random_lqr_kkt(3, 1, 4, 2, seed=1, mid_p=1, hess_mode=1, explicit_D2=True)
    f, ins = _abi_args(prob)
    n, m, N, b = 3, 1, 4, 2
    NN, P = N * n + (N - 1) * m, int(f["p"].sum()) + (N - 1) * n
    sol = [np.zeros((b, NN)), np.zeros((b, P)), np.ones((b, NN)), np.ones((b, P))]
    outs = _abi_grads(f, dense=True, d2x=True)
    L = _lib.lib()
    p0 = np.ascontiguousarray(f["p"], dtype=np.int32)

    def rc(hp=True, n_=n, m_=m, N_=N, b_=b, p=p0, hess=1, flags=0, drop=(), keep=None):
        args = [_lib.ptr(a) for a in ins] + [_lib.ptr(a) for a in sol]
        for i in drop:
            args[i] = None
        g = [_lib.ptr(a) if (keep is None or i in keep) else None for i, a in enumerate(outs)]
        if keep is None:
            g[2] = None  # gHux: this problem is not DENSE
        return L.lqrb_kkt_grad_f64(handle._h if hp else None, n_, m_, N_, b_, None if p is None else p.ctypes.data,
                                   hess, flags, *args, *g, None)
    assert rc() == 0
    assert rc(hp=False) == -1
    assert rc(n_=0) == -2 and rc(n_=129) == -2
    assert rc(m_=0) == -3 and rc(m_=n + 1) == -3
    assert rc(N_=1) == -4
    assert rc(b_=-1) == -5
    assert rc(p=None) == -6 and rc(p=np.array([3, -1, 0, 3], dtype=np.int32)) == -6
    assert rc(hess=3) == -7
    assert rc(flags=_lib.FLAG_SOC) == -8 and rc(flags=_lib.FLAG_LTI) == -8
    for i, code in ((0, -9), (1, -10), (3, -12), (4, -13), (6, -15), (7, -16), (8, -17)):
        assert rc(drop=(i,)) == code, code
    assert rc(drop=(2,)) == 0  # Hux may be NULL
    assert rc(drop=(9,)) == 0 and rc(drop=(10,)) == 0  # either cotangent may be NULL
    assert rc(drop=(9, 10)) == -18
    assert rc(keep=()) == -20
    assert rc(keep=(2,)) == -22  # gHux needs LQRB_HESS_DENSE
    assert rc(keep=(2,), hess=0) == 0
    assert rc(drop=(5,), keep=(8,)) == -28  # gD2 needs an explicit D2
    p_none = np.array([0, 0, 0, 0], dtype=np.int32)
    assert rc(p=p_none, drop=(6,), keep=(9,)) == -29 and rc(p=p_none, drop=(6,), keep=(10,)) == -30


def test_indefinite_instance_reports_info_and_leaves_neighbours(handle):
    prob = problems.random_lqr_kkt(6, 3, 10, 7, seed=4, mid_p=1)
    dz, mult, dzb, mb, g = _solve_and_grad(handle, prob, seed=2)
    bad = {k: (np.array(v, copy=True) if isinstance(v, np.ndarray) else v) for k, v in prob.items()}
    bad["R"][3] = -bad["R"][3]
    gb, info = ops.kkt_grad_problem(bad, dz, mult, dzb, mb, handle=handle)
    assert info[3] != 0 and (np.delete(info, 3) == 0).all(), info
    keep = [i for i in range(7) if i != 3]
    for k in NAMES:
        if isinstance(g[k], list):
            for x, y in zip(gb[k], g[k]):
                assert np.array_equal(x[keep], y[keep]), k
        elif g[k] is not None:
            assert np.array_equal(gb[k][keep], g[k][keep]), k


def test_run_to_run_determinism(handle):
    prob = problems.random_lqr_kkt(12, 4, 30, 70, seed=8, mid_p=2)
    dz, mult, dzb, mb, g1 = _solve_and_grad(handle, prob, seed=8)
    g2, _ = ops.kkt_grad_problem(prob, dz, mult, dzb, mb, handle=handle)
    for k in NAMES:
        assert np.array_equal(_flat(g1[k]), _flat(g2[k])), k


def test_kept_factorisation_and_condition_record_are_left_alone(handle):
    """A grad call between lqrb_kkt_factor_f64 and lqrb_kkt_solve_factored_f64 does not replace the kept factor, and
    lqrb_kkt_last_condition keeps reporting the last forward solve."""
    fp = problems.random_lqr_kkt(6, 2, 9, 4, seed=2, mid_p=1)
    f = ops.kkt_flatten(fp)
    n, m, N, b, p = 6, 2, 9, 4, f["p"]
    ops.kkt_factor(handle, n, m, N, b, p, 1, 0, f["Q"], f["R"], None, f["A"], f["B"], None, f["C"])
    NN, P = N * n + (N - 1) * m, int(p.sum()) + (N - 1) * n

    def factored():
        dz, mult = np.zeros((b, NN)), np.zeros((b, P))
        ops.kkt_solve_factored(handle, n, m, N, b, p, 1, 0, 0, f["q"], f["r"], f["d"], f["c"], dz, mult)
        return dz, mult
    before = factored()
    tuned = problems.random_lqr_kkt(12, 4, 20, 5, seed=3)  # a tuned kernel keeps a conditioning record
    dz, mult, info = ops.kkt_solve_problem(tuned, handle=handle)
    bits, resolved = handle.kkt_last_condition(5)
    other = problems.random_lqr_kkt(12, 4, 20, 9, seed=4, mid_p=1)
    odz, omult, _ = ops.kkt_solve_problem(other, handle=handle)
    bits_o, _ = handle.kkt_last_condition(9)
    ops.kkt_solve_problem(tuned, handle=handle)
    ops.kkt_grad_problem(other, odz, omult, np.ones_like(odz), np.ones_like(omult), handle=handle)
    bits2, resolved2 = handle.kkt_last_condition(9)
    assert (bits_o >= 0).all()  # `other` runs a tuned kernel: a record kept by the grad call would track 9 instances
    assert np.array_equal(bits2[:5], bits) and (bits2[5:] == -1).all() and resolved2 == resolved
    after = factored()
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])


def _torch_leaves(prob, dense):
    import torch
    t = {k: torch.tensor(prob[k], device="cuda", requires_grad=True) for k in ("Q", "R", "q", "r", "A", "B", "d")}
    t["C"] = [torch.tensor(x, device="cuda", requires_grad=True) for x in prob["C"]]
    t["c"] = [torch.tensor(x, device="cuda", requires_grad=True) for x in prob["c"]]
    t["Hux"] = torch.tensor(prob["Hux"], device="cuda", requires_grad=True) if dense else None
    return t


@pytest.mark.parametrize("hess", [1, 0])
def test_autograd_gradcheck(hess):
    import torch
    from lqr_b200.autograd import kkt_solve
    n, m, N, b = 3, 2, 5, 2
    prob = problems.random_lqr_kkt(n, m, N, b, seed=6, dt=0.1, mid_p=1, hess_mode=hess)
    prob["A"] = np.repeat(prob["A"][:1], b, axis=0)  # one A for the whole batch, broadcast below
    t = _torch_leaves(prob, hess == 0)
    t["A"] = torch.tensor(prob["A"][:1], device="cuda", requires_grad=True)
    plain = ["Q", "R", "q", "r", "A", "B", "d"] + (["Hux"] if hess == 0 else [])
    xs = [t[k] for k in plain] + t["C"] + t["c"]

    def f(*xs):
        kw = dict(zip(plain, xs[:len(plain)]))
        C, c = list(xs[len(plain):len(plain) + N]), list(xs[len(plain) + N:])
        X, U, mult, info = kkt_solve(kw["Q"], kw["R"], kw["q"], kw["r"], kw["A"], kw["B"], kw["d"], C, c,
                                     Hux=kw.get("Hux"), hess_mode=hess)
        return X, U, mult
    # Central differences of a forward solve with absolute error e carry rounding noise up to e / eps (and a
    # truncation error of order eps^2, negligible at eps = 1e-6).  e is the library's forward error against the
    # refined solve, largest over this problem and 16 neighbours one step away (it varies from point to point; doubled
    # for the points gradcheck visits that were not sampled), and the tolerance is that noise bound, never below 1e-7.
    # Entries whose true derivative is zero (the states pinned by the initial-condition rows) see nothing but noise.
    from oracle import dense_kkt

    def forward_error(p):
        dz, mult, _ = ops.kkt_solve_problem(p)
        return max(max(np.abs(dz[i] - zt).max(), np.abs(mult[i] - lt).max())
                   for i, (zt, lt) in enumerate(dense_kkt.kkt_truth(p, i) for i in range(b)))

    def neighbour(h, seed):
        rng, p = np.random.default_rng(seed), dict(prob)
        for k in plain:
            p[k] = prob[k] + h * rng.choice([-1.0, 1.0], np.shape(prob[k]))
            if k in ("Q", "R"):  # the solve reads the upper triangle, the refined solve the whole matrix
                p[k] = 0.5 * (p[k] + np.swapaxes(p[k], -1, -2))
        for k in ("C", "c"):
            p[k] = [x + h * rng.choice([-1.0, 1.0], x.shape) for x in prob[k]]
        return p
    eps = 1e-6
    err = 2 * max(forward_error(prob), *(forward_error(neighbour(eps, s)) for s in range(16)))
    assert torch.autograd.gradcheck(f, tuple(xs), eps=eps, atol=max(1e-7, err / eps), rtol=1e-6)


def test_autograd_matches_library_and_rejects_cpu(handle):
    import torch
    from lqr_b200.autograd import kkt_solve
    prob = problems.random_lqr_kkt(8, 2, 15, 4, seed=12, mid_p=1, explicit_D2=True)
    t = _torch_leaves(prob, False)
    t["D2"] = [torch.tensor(x, device="cuda", requires_grad=True) for x in prob["D2"]]
    X, U, mult, info = kkt_solve(t["Q"], t["R"], t["q"], t["r"], t["A"], t["B"], t["d"], t["C"], t["c"], D2=t["D2"])
    assert (info == 0).all() and not info.requires_grad
    WX, WU, Wm = (torch.randn(x.shape, dtype=torch.float64, device="cuda") for x in (X, U, mult))
    ((X * WX).sum() + (U * WU).sum() + (mult * Wm).sum()).backward()
    dz, mult_np, _ = ops.kkt_solve_problem(prob, handle=handle)
    b, N, n, m = 4, 15, 8, 2
    dzb = np.zeros_like(dz)
    body = dzb[:, :(N - 1) * (n + m)].reshape(b, N - 1, n + m)
    body[:, :, :n] = WX[:, :N - 1].cpu().numpy()
    body[:, :, n:] = WU.cpu().numpy()
    dzb[:, (N - 1) * (n + m):] = WX[:, N - 1].cpu().numpy()
    g, _ = ops.kkt_grad_problem(prob, dz, mult_np, dzb, Wm.cpu().numpy(), handle=handle)
    # autograd symmetrises Q, R first: its gradient is the symmetric part of the ABI's (already symmetric) one
    for k in ("Q", "R", "q", "r", "A", "B", "d"):
        np.testing.assert_allclose(t[k].grad.cpu().numpy(), g[k], rtol=1e-11, atol=1e-13)
    for k in ("C", "c", "D2"):
        for x, y in zip(t[k], g[k]):
            np.testing.assert_allclose(x.grad.cpu().numpy(), y, rtol=1e-11, atol=1e-13)
    with pytest.raises(TypeError):
        kkt_solve(*(torch.tensor(prob[k]) for k in ("Q", "R", "q", "r", "A", "B", "d")),
                  [torch.tensor(x) for x in prob["C"]], [torch.tensor(x) for x in prob["c"]])


def test_autograd_calls_on_two_streams_are_ordered():
    """kkt_solve calls share the device's handle and its scratch.  A call issued on stream s2 while the previous call,
    on s1, has not even started (s1 is held by a sleep kernel) must wait for it: checked by the order in which the two
    streams reach their end events and by the values of both calls against the same problems solved one by one."""
    import torch
    from lqr_b200.autograd import kkt_solve
    ps = [problems.random_lqr_kkt(12, 4, 40, 64, seed=s, mid_p=1) for s in (13, 14)]

    def run(t):
        X, U, mult, _ = kkt_solve(t["Q"], t["R"], t["q"], t["r"], t["A"], t["B"], t["d"], t["C"], t["c"])
        (X.square().sum() + U.sum() + mult.sum()).backward()
        return [X.detach(), mult.detach()] + [t[k].grad for k in ("Q", "R", "q", "r", "A", "B", "d")] + \
            [x.grad for x in t["C"]]
    ref = [run(_torch_leaves(p, False)) for p in ps]
    ins = [_torch_leaves(p, False) for p in ps]  # made before the streams below: a pageable copy would wait for the sleep
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    e1, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s1):
        torch.cuda._sleep(1_000_000_000)  # about half a second of the GPU clock
        out1 = run(ins[0])
        e1.record()
    with torch.cuda.stream(s2):
        out2 = run(ins[1])
        e2.record()
    torch.cuda.synchronize()
    assert e1.elapsed_time(e2) >= 0, "the call on s2 finished before the earlier call on s1"
    for got, want in zip(out1 + out2, ref[0] + ref[1]):
        assert torch.equal(got, want)


def test_autograd_has_no_double_backward():
    import torch
    from lqr_b200.autograd import kkt_solve
    prob = problems.random_lqr_kkt(4, 2, 6, 2, seed=3, mid_p=1)
    t = _torch_leaves(prob, False)
    X, U, mult, _ = kkt_solve(t["Q"], t["R"], t["q"], t["r"], t["A"], t["B"], t["d"], t["C"], t["c"])
    (gA,) = torch.autograd.grad(X.square().sum() + mult.square().sum(), t["A"], create_graph=True)
    with pytest.raises(RuntimeError):
        gA.sum().backward()
