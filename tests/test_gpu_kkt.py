"""GPU parity: batched constrained KKT solve (C ABI -> CUDA) against the CPU oracle (the reference's
block algorithm) and the refined global KKT solve, on the reference's fixtures and the configs.

Tolerances (SURVEY §8d): relative error of dz and of the multipliers, stationarity residual and
primal residual all <= 1e-10 unless a per-case value is written below."""
import numpy as np
import pytest

from lqr_b200 import ops, problems

pytestmark = pytest.mark.gpu
TOL = 1e-10


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _check(prob, handle, oracle_mod, tol=TOL, truth_instances=(0,), soc=False, res_tol=TOL):
    from oracle import dense_kkt
    dz, lam, info, res = ops.kkt_solve_problem(prob, soc=soc, want_res=True, handle=handle)
    dzo, lamo, infoo, reso = oracle_mod.kkt_solve(prob, soc=soc, want_res=True)
    assert (info == 0).all() and (infoo == 0).all(), handle.last_kernel
    b = dz.shape[0]
    for i in range(b):
        assert _rel(dz[i], dzo[i]) <= tol, (i, _rel(dz[i], dzo[i]), handle.last_kernel)
        assert _rel(lam[i], lamo[i]) <= tol, (i, _rel(lam[i], lamo[i]), handle.last_kernel)
        assert np.linalg.norm(res[i] - reso[i]) <= tol * max(1.0, np.linalg.norm(reso[i]))
    for i in truth_instances:
        zt, lt = dense_kkt.kkt_truth(prob, i, soc=soc)
        assert _rel(dz[i], zt) <= tol and _rel(lam[i], lt) <= tol
        rs, rp = dense_kkt.kkt_residuals(prob, i, dz[i], lam[i], soc=soc)
        assert rs <= res_tol and rp <= res_tol, (rs, rp)
    return dz, lam


def test_config1_cartpole_fixture(handle, oracle_mod):
    """config 1: single cartpole instance, block-Cholesky vs sparse/dense KKT (test/cartpole.jl)."""
    _check(problems.cartpole_fixture(), handle, oracle_mod)
    assert handle.last_kernel.startswith("kkt_tpi<4,1")


@pytest.mark.parametrize("dense_cost", [False, True])
def test_double_integrator_fixture(handle, oracle_mod, dense_cost):
    """test/cholesky_solve.jl:7-44 on DoubleIntegrator(3,101): ||D dz + d||, ||H dz + g + D'lam|| and
    equality with the dense KKT solve."""
    _check(problems.double_integrator_fixture(dense_cost=dense_cost), handle, oracle_mod)
    assert handle.last_kernel.startswith("kkt_tpi<6,3")


def test_second_order_correction_chain(handle, oracle_mod):
    """Ginv=false chain (src/cholesky_solver.jl:254-273): dz = -D'(DD')^-1 d.  cond(DD') of the double
    integrator is ~1e7, so this case is held to 1e-8."""
    _check(problems.cartpole_fixture(), handle, oracle_mod, soc=True)
    _check(problems.double_integrator_fixture(), handle, oracle_mod, soc=True, tol=1e-8, res_tol=1e-8)


@pytest.mark.parametrize("mid_p", [0, 1])
@pytest.mark.parametrize("batch", [1, 33, 130])
def test_config3_dubins(handle, oracle_mod, mid_p, batch):
    prob = problems.dubins_kkt_batch(batch, seed=batch, N=201, mid_p=mid_p)
    _check(prob, handle, oracle_mod, truth_instances=(0, batch - 1))
    assert handle.last_kernel.startswith("kkt_tpi<3,2")


@pytest.mark.parametrize("hess", [0, 1, 2])
@pytest.mark.parametrize("n,m,N,mid_p", [(2, 1, 9, 0), (4, 2, 9, 1), (4, 1, 30, 0), (3, 2, 6, 0), (6, 3, 12, 1), (4, 2, 12, 0),
                                        (6, 3, 14, 0), (2, 2, 9, 0), (2, 2, 10, 1), (3, 1, 12, 0), (3, 3, 9, 0), (3, 3, 11, 1),
                                        (5, 1, 14, 0), (6, 1, 15, 0), (5, 2, 12, 0), (5, 2, 13, 1), (6, 2, 14, 0), (6, 2, 15, 1),
                                        (4, 3, 9, 0), (4, 3, 10, 1), (5, 3, 11, 0), (5, 3, 12, 1)])
def test_tpi_hessian_modes(handle, oracle_mod, n, m, N, mid_p, hess):
    prob = problems.random_lqr_kkt(n, m, N, 37, seed=7 * n + hess, mid_p=mid_p, hess_mode=hess)
    _check(prob, handle, oracle_mod)
    assert handle.last_kernel.startswith("kkt_tpi")


@pytest.mark.parametrize("hess", [0, 1, 2])
@pytest.mark.parametrize("n,m,N,mid_p,d2x", [(7, 2, 10, 1, False), (4, 1, 12, 0, True), (3, 2, 8, 1, True),
                                            (10, 3, 40, 0, False), (12, 4, 9, 2, True), (20, 6, 6, 0, False),
                                            (4, 4, 2, 0, False)])
def test_cooperative_kernel(handle, oracle_mod, n, m, N, mid_p, d2x, hess):
    prob = problems.random_lqr_kkt(n, m, N, 6, seed=n + hess, mid_p=mid_p, hess_mode=hess, explicit_D2=d2x)
    handle.set_option("kkt_pad", 0)  # (without it most of these shapes are embedded in a tuned size class, see below)
    try:
        _check(prob, handle, oracle_mod)
    finally:
        handle.set_option("kkt_pad", 1)
    assert handle.last_kernel.startswith("kkt_coop")


@pytest.mark.parametrize("hess", [0, 1, 2])
@pytest.mark.parametrize("n,m,N,batch,mid_p,kern", [
    (7, 2, 12, 6, 1, "kkt_wp_dmma<8,3"), (10, 3, 40, 33, 0, "kkt_wp_dmma<12,4|kkt_hw<12,4"), (9, 2, 30, 5, 1, "kkt_wp_dmma<12,3"),
    (5, 3, 14, 7, 2, "kkt_wp_dmma<8,4"), (7, 3, 21, 34, 2, "kkt_wp_dmma<8,4"), (11, 1, 25, 4, 0, "kkt_wp_dmma<12,2|kkt_hw<12,4"),
    (14, 7, 12, 5, 0, "kkt_cta_dmma<16,8"), (20, 6, 14, 3, 2, "kkt_cta_dmma<24,8"), (13, 4, 20, 6, 1, "kkt_cta_dmma<16,8"),
    (30, 8, 12, 3, 0, "kkt_cta_dmma<32,16"), (40, 12, 11, 2, 1, "kkt_cta_dmma<48,16"), (60, 10, 12, 2, 0, "kkt_cta_dmma<64,16"),
    (16, 5, 18, 4, 3, "kkt_cta_dmma<16,8")])
def test_shapes_without_a_tuned_kernel_are_padded_into_one(handle, oracle_mod, n, m, N, batch, mid_p, kern, hess):
    """A shape that has no tuned kernel of its own is embedded in the next tuned size class (decoupled pad states and
    controls whose solution is exactly zero) instead of falling to the general kernel; the outputs are the original
    problem's.  Dense Hessians stay on the general kernel above n = 12 (the CTA kernels do not have that mode)."""
    from oracle import dense_kkt
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=5 * n + m + hess, mid_p=mid_p, hess_mode=hess)
    dz, lam, info, res = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
    if hess == 0 and n > 12:
        assert handle.last_kernel.startswith("kkt_coop")
    else:
        assert any(handle.last_kernel.startswith(k) for k in kern.split("|")), handle.last_kernel
        assert handle.last_kernel.endswith(f"<- ({n},{m}) padded"), handle.last_kernel
    dzo, lamo, infoo, reso = oracle_mod.kkt_solve(prob, want_res=True)
    assert (info == 0).all() and (infoo == 0).all()
    for i in range(batch):
        zt, lt = dense_kkt.kkt_truth(prob, i)
        tol = max(TOL, 4.0 * max(_rel(dzo[i], zt), _rel(lamo[i], lt)))
        assert _rel(dz[i], zt) <= tol and _rel(lam[i], lt) <= tol, (i, tol, _rel(dz[i], zt), _rel(lam[i], lt))
        assert np.linalg.norm(res[i] - reso[i]) <= 2 * tol * max(1.0, np.linalg.norm(reso[i]))
        rs, rp = dense_kkt.kkt_residuals(prob, i, dz[i], lam[i])
        assert rs <= 10 * TOL and rp <= 10 * TOL, (rs, rp)


# kkt_variant: 0 = default (half warp per instance), 5 = warp per instance on the FP64 tensor cores (the default only
# for the shapes the half-warp kernel does not have: odd m, dense Hessian)
QUAD_VARIANTS = [(0, "kkt_hw<"), (5, "kkt_wp_dmma<")]


@pytest.mark.parametrize("variant,kern", QUAD_VARIANTS)
@pytest.mark.parametrize("n,m,N,batch", [(12, 4, 40, 6), (12, 4, 8, 5), (12, 4, 6, 1), (8, 4, 25, 7), (8, 4, 4, 3), (12, 4, 301, 9),
                                         (12, 4, 1001, 2)])
def test_half_warp_kernel(handle, oracle_mod, n, m, N, batch, variant, kern):
    """config 5a-K shape: init + dynamics + goal, block-diagonal Hessian -> warp- / half-warp-per-instance kernels."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=n + N, mid_p=0, hess_mode=1)
    handle.set_option("kkt_variant", variant)
    try:
        _check(prob, handle, oracle_mod, truth_instances=(0, batch - 1))
        assert handle.last_kernel.startswith(kern)
    finally:
        handle.set_option("kkt_variant", 0)


@pytest.mark.parametrize("hess", [1, 2])
@pytest.mark.parametrize("soc", [False, True])
@pytest.mark.parametrize("n,m,N,batch,kern,variant", [(12, 4, 40, 6, "kkt_wp_dmma<", 5), (8, 4, 21, 5, "kkt_wp_dmma<", 5),
                                                      (12, 1, 40, 4, "kkt_wp_dmma<", 0), (8, 1, 25, 3, "kkt_wp_dmma<", 0),
                                                      (12, 4, 40, 6, "kkt_hw<", 0), (8, 4, 21, 5, "kkt_hw<", 0),
                                                      (64, 16, 12, 2, "kkt_cta_dmma<", 0)])
def test_tuned_kernels_hessian_modes_and_soc(handle, oracle_mod, n, m, N, batch, kern, variant, hess, soc):
    """Diagonal / block-diagonal BlockCholesky modes (src/block_cholesky.jl:69-91) and the Ginv=false chain of
    second_order_correction! (src/cholesky_solver.jl:254-273) on the tuned large-size kernels."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=3 * n + hess, mid_p=0, hess_mode=hess)
    handle.set_option("kkt_variant", variant)
    try:
        _check(prob, handle, oracle_mod, soc=soc, tol=1e-9 if soc else TOL, res_tol=1e-9 if soc else TOL)
        assert handle.last_kernel.startswith(kern) and (",soc" in handle.last_kernel) == soc
    finally:
        handle.set_option("kkt_variant", 0)


def test_half_warp_matches_cooperative_kernel(handle):
    prob = problems.random_lqr_kkt(12, 4, 120, 11, seed=5, mid_p=0, hess_mode=1)
    dz1, lam1, i1, r1 = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
    assert handle.last_kernel.startswith("kkt_hw<")
    handle.set_option("kkt_variant", 2)
    try:
        dz2, lam2, i2, r2 = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
        assert handle.last_kernel.startswith("kkt_coop")
    finally:
        handle.set_option("kkt_variant", 0)
    assert (i1 == 0).all() and (i2 == 0).all()
    assert _rel(dz1, dz2) <= 1e-11 and _rel(lam1, lam2) <= 1e-11
    assert np.abs(r1 - r2).max() <= 1e-10 * max(1.0, np.abs(r2).max())


def test_half_warp_info_flags(handle):
    prob = problems.random_lqr_kkt(12, 4, 30, 5, seed=9, mid_p=0, hess_mode=1)
    prob["R"][2, 7] = -np.eye(4)
    for variant, kern in ((0, "kkt_hw<"), (5, "kkt_wp_dmma<")):
        handle.set_option("kkt_variant", variant)
        try:
            _, _, info = ops.kkt_solve_problem(prob, handle=handle)
        finally:
            handle.set_option("kkt_variant", 0)
        assert handle.last_kernel.startswith(kern)
        assert info[2] == 8 * 1000 + 12 + 1 and (np.delete(info, 2) == 0).all(), (kern, info)


def test_irregular_stage_pattern(handle, oracle_mod):
    """A waypoint constraint on a single interior knot: p is not [P1, PM.., PN] -> padded into the warp-per-instance
    kernel (per-knot stage rows); with kkt_pad = 0 the cooperative kernel."""
    prob = problems.random_lqr_kkt(4, 1, 16, 5, seed=3, mid_p=1)
    p = prob["p"].copy()
    for k in range(1, 15):
        if k != 8:
            p[k] = 0
            prob["C"][k] = np.zeros((5, 0, 5))
            prob["c"][k] = np.zeros((5, 0))
    prob["p"] = p
    _check(prob, handle, oracle_mod)
    assert handle.last_kernel.startswith("kkt_wp_dmma<8,2,p=8/per-knot<=1/8") and "(4,1) padded" in handle.last_kernel
    handle.set_option("kkt_pad", 0)
    try:
        _check(prob, handle, oracle_mod)
    finally:
        handle.set_option("kkt_pad", 1)
    assert handle.last_kernel.startswith("kkt_coop")


def test_large_dense_schur_variant(handle, oracle_mod):
    """config 5b shape (n=64, m=16) at a short horizon: 1e-10 against the extended-precision solve, or 4x the error
    the reference's own operation order (the CPU oracle) makes on this input if that is larger (measured here)."""
    from oracle import dense_kkt
    prob = problems.random_lqr_kkt(64, 16, 6, 2, seed=4)
    dz, lam, info = ops.kkt_solve_problem(prob, handle=handle)
    assert handle.last_kernel.startswith("kkt_cta_dmma<64,16") and (info == 0).all()
    dzo, lamo, _ = oracle_mod.kkt_solve(prob)
    for i in range(2):
        zt, lt = dense_kkt.kkt_truth(prob, i)
        tol = max(TOL, 4.0 * max(_rel(dzo[i], zt), _rel(lamo[i], lt)))
        assert _rel(dz[i], zt) <= tol and _rel(lam[i], lt) <= tol, (i, tol)
        rs, rp = dense_kkt.kkt_residuals(prob, i, dz[i], lam[i])
        assert rs <= TOL and rp <= TOL, (rs, rp)


@pytest.mark.parametrize("N,batch", [(12, 3), (101, 2), (30, 5)])
def test_cta_dmma_kernel(handle, oracle_mod, N, batch):
    """config 5b-K: CTA-per-instance FP64 tensor-core kernel + parallel pre-pass."""
    prob = problems.random_lqr_kkt(64, 16, N, batch, seed=N, mid_p=0, hess_mode=1)
    _check(prob, handle, oracle_mod, truth_instances=(0,))
    assert handle.last_kernel.startswith("kkt_cta_dmma<64,16")


@pytest.mark.parametrize("hess,soc", [(1, False), (2, False), (1, True)])
@pytest.mark.parametrize("n,m,N,batch", [(16, 8, 24, 5), (24, 8, 18, 3), (32, 8, 30, 4), (48, 16, 16, 3), (16, 16, 12, 5),
                                         (24, 16, 14, 3), (32, 16, 15, 4)])
def test_cta_dmma_other_sizes(handle, oracle_mod, n, m, N, batch, hess, soc):
    """The CTA-per-instance tensor-core KKT kernel at the other sizes of the Riccati CTA family
    (n = 16, 24, 32, 48: 2, 3, 4, 6 warps), against the oracle and against the cooperative kernel."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=7 * n + hess, mid_p=0, hess_mode=hess)
    _check(prob, handle, oracle_mod, soc=soc, tol=1e-9 if soc else TOL, res_tol=1e-9 if soc else TOL)
    assert handle.last_kernel.startswith(f"kkt_cta_dmma<{n},{m}") and (",soc" in handle.last_kernel) == soc
    dz1, lam1, i1 = ops.kkt_solve_problem(prob, soc=soc, handle=handle)
    handle.set_option("kkt_variant", 2)
    try:
        dz2, lam2, i2 = ops.kkt_solve_problem(prob, soc=soc, handle=handle)
        assert handle.last_kernel.startswith("kkt_coop")
    finally:
        handle.set_option("kkt_variant", 0)
    assert (i1 == 0).all() and (i2 == 0).all()
    assert _rel(dz1, dz2) <= 1e-9 and _rel(lam1, lam2) <= 1e-9


def test_cta_dmma_matches_cooperative_kernel(handle):
    prob = problems.random_lqr_kkt(64, 16, 20, 3, seed=6, mid_p=0, hess_mode=1)
    dz1, lam1, i1, r1 = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
    assert handle.last_kernel.startswith("kkt_cta_dmma")
    handle.set_option("kkt_variant", 2)
    try:
        dz2, lam2, i2, r2 = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
        assert handle.last_kernel.startswith("kkt_coop")
    finally:
        handle.set_option("kkt_variant", 0)
    assert (i1 == 0).all() and (i2 == 0).all()
    assert _rel(dz1, dz2) <= 1e-10 and _rel(lam1, lam2) <= 1e-10
    assert np.abs(r1 - r2).max() <= 1e-9 * max(1.0, np.abs(r2).max())


def test_cta_dmma_info_flags(handle):
    prob = problems.random_lqr_kkt(64, 16, 10, 3, seed=9, mid_p=0, hess_mode=1)
    prob["Q"][1, 4] = -np.eye(64)
    _, _, info = ops.kkt_solve_problem(prob, handle=handle)
    assert handle.last_kernel.startswith("kkt_cta_dmma")
    assert info[1] == 5 * 1000 + 1 and (np.delete(info, 1) == 0).all()


def test_info_flags_bad_hessian(handle):
    prob = problems.dubins_kkt_batch(40, seed=1, N=21)
    prob["R"][5, 3] = -np.eye(2)
    _, _, info = ops.kkt_solve_problem(prob, handle=handle)
    assert info[5] == 4 * 1000 + 3 + 1 and (np.delete(info, 5) == 0).all()


def test_idempotent_full_width_batch(handle):
    """Size-independent check at a large batch: the step computed from the solution point has zero
    primal residual (D dz + d = 0 row by row), evaluated block-wise on the host for every instance."""
    b = 4096
    prob = problems.dubins_kkt_batch(b, seed=2, N=201)
    dz, lam, info = ops.kkt_solve_problem(prob, handle=handle)
    assert (info == 0).all()
    n, m, N = 3, 2, 201
    X, U = ops.split_primals(dz, n, m, N)
    dyn = np.einsum("bkij,bkj->bki", prob["A"], X[:, :-1]) + np.einsum("bkij,bkj->bki", prob["B"], U) \
        - X[:, 1:] + prob["d"]
    assert np.abs(dyn).max() <= 1e-10
    assert np.abs(X[:, 0] + prob["c"][0]).max() <= 1e-10
    assert np.abs(X[:, -1] + prob["c"][-1]).max() <= 1e-10


def _kkt_residuals_all(prob, dz, lam):
    """Stationarity and primal residuals of every instance (init + dynamics + goal pattern), host einsum."""
    n, m, N = prob["n"], prob["m"], prob["N"]
    X, U = ops.split_primals(dz, n, m, N)
    p = prob["p"]
    assert p[0] == n and p[-1] == n and all(v == 0 for v in p[1:-1])
    mu0, mu_last = lam[:, :n], lam[:, -n:]
    L = lam[:, n:-n].reshape(lam.shape[0], N - 1, n)          # lam_0 .. lam_{N-2}
    A, B, Q, R = prob["A"], prob["B"], prob["Q"], prob["R"]
    dyn = np.einsum("bkij,bkj->bki", A, X[:, :-1]) + np.einsum("bkij,bkj->bki", B, U) - X[:, 1:] + prob["d"]
    C0, CN = prob["C"][0], prob["C"][-1]
    z0 = np.concatenate([X[:, 0], U[:, 0]], axis=1)
    prim = max(np.abs(dyn).max(), np.abs(np.einsum("bij,bj->bi", C0, z0) + prob["c"][0]).max(),
               np.abs(np.einsum("bij,bj->bi", CN, X[:, -1]) + prob["c"][-1]).max())
    sx = np.einsum("bkij,bkj->bki", Q, X) + prob["q"]
    sx[:, :-1] += np.einsum("bkji,bkj->bki", A, L)
    sx[:, 1:] -= L
    sx[:, 0] += np.einsum("bji,bj->bi", C0[:, :, :n], mu0)
    sx[:, -1] += np.einsum("bji,bj->bi", CN, mu_last)
    su = np.einsum("bkij,bkj->bki", R, U) + prob["r"] + np.einsum("bkji,bkj->bki", B, L)
    su[:, 0] += np.einsum("bji,bj->bi", C0[:, :, n:], mu0)
    scale = max(1.0, np.abs(prob["q"]).max(), np.abs(lam).max())
    return max(np.abs(sx).max(), np.abs(su).max()) / scale, prim


@pytest.mark.parametrize("n,m,N,batch,kern", [(12, 4, 101, 2049, "kkt_hw<"), (64, 16, 41, 300, "kkt_cta_dmma<")])
def test_tuned_kernels_kkt_conditions_at_scale(handle, n, m, N, batch, kern):
    """Size-independent property on a batch that spans many CTAs (and an odd tail): the returned step and
    multipliers satisfy the KKT conditions  H dz + g + D'lam = 0,  D dz + d = 0  for EVERY instance."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=11, mid_p=0, hess_mode=1)
    dz, lam, info = ops.kkt_solve_problem(prob, handle=handle)
    assert handle.last_kernel.startswith(kern) and (info == 0).all()
    stat, prim = _kkt_residuals_all(prob, dz, lam)
    assert stat <= 1e-10 and prim <= 1e-10, (stat, prim)


@pytest.mark.parametrize("n,m,N,batch", [(12, 4, 30, 9000), (64, 16, 8, 700)])
def test_tuned_kernels_chunked_scratch(handle, n, m, N, batch):
    """The tuned kernels process the batch in chunks when their scratch would exceed `scratch_budget_mb`;
    a tiny budget forces several chunks (one resident wave each) and must reproduce the one-chunk result."""
    prob = problems.random_lqr_kkt(n, m, N, 64, seed=5, mid_p=0, hess_mode=1)
    rep = (batch + 63) // 64
    big = {k: (np.tile(v, (rep,) + (1,) * (v.ndim - 1))[:batch] if isinstance(v, np.ndarray) and v.ndim > 1 else v)
           for k, v in prob.items()}
    big["C"] = [np.tile(c, (rep, 1, 1))[:batch] for c in prob["C"]]
    big["c"] = [np.tile(c, (rep, 1))[:batch] for c in prob["c"]]
    dz1, lam1, i1 = ops.kkt_solve_problem(big, handle=handle)
    handle.set_option("scratch_budget_mb", 1)
    try:
        dz2, lam2, i2 = ops.kkt_solve_problem(big, handle=handle)
    finally:
        handle.set_option("scratch_budget_mb", 49152)
    assert (i1 == 0).all() and (i2 == 0).all()
    assert np.array_equal(dz1, dz2) and np.array_equal(lam1, lam2)
    assert np.array_equal(dz1[:64], dz1[64:128])      # replicated instances give replicated answers


@pytest.mark.parametrize("soc", [False, True])
@pytest.mark.parametrize("n,m,N,batch", [(12, 4, 40, 6), (8, 4, 21, 5), (12, 1, 40, 3), (8, 1, 30, 4), (12, 4, 301, 2)])
def test_dense_hessian_on_the_tensor_core_kernel(handle, oracle_mod, n, m, N, batch, soc):
    """Whole-matrix BlockCholesky mode (Hux != 0, src/block_cholesky.jl:55-66) at the quadrotor sizes: lands on the
    warp-per-instance tensor-core kernel (H^-1 is a z-space inverse there), not on the cooperative fallback."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=5 * n + m, mid_p=0, hess_mode=0)
    assert np.abs(prob["Hux"]).max() > 0
    _check(prob, handle, oracle_mod, soc=soc, tol=1e-9 if soc else TOL, res_tol=1e-9 if soc else TOL,
           truth_instances=(0, batch - 1))
    assert handle.last_kernel.startswith(f"kkt_wp_dmma<{n},{m}") and ",hess=0" in handle.last_kernel


@pytest.mark.parametrize("hess,soc", [(1, False), (2, False), (0, False), (1, True)])
@pytest.mark.parametrize("n,m,N,batch,mid_p", [(12, 4, 40, 7, 1), (12, 4, 41, 6, 2), (8, 4, 30, 5, 1), (12, 4, 25, 3, 3),
                                               (8, 4, 31, 4, 2), (8, 4, 40, 3, 3)])
def test_stage_constraints_on_the_tensor_core_kernel(handle, oracle_mod, n, m, N, batch, mid_p, hess, soc):
    """Mid-horizon stage constraints (the reference's DoubleIntegrator pattern p = [n, ps, ..., ps, n],
    test/problems.jl:39-43) at the quadrotor sizes run on the warp-per-instance tensor-core kernel — ps <= 4 rows per
    knot as vector work next to the n x n blocks — not on the cooperative fallback.  Odd ps puts knot records on odd
    doubles (the bulk copies then start one double early): batches > 1 and both parities of N cover that."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=11 * n + mid_p, mid_p=mid_p, hess_mode=hess)
    _check(prob, handle, oracle_mod, soc=soc, tol=1e-9 if soc else TOL, res_tol=1e-9 if soc else TOL,
           truth_instances=(0, batch - 1))
    assert handle.last_kernel.startswith(f"kkt_wp_dmma<{n},{m},p={n}/{mid_p}/{n}"), handle.last_kernel


@pytest.mark.parametrize("hess", [0, 1, 2])
@pytest.mark.parametrize("n,m,N,batch,mid_p", [(12, 3, 40, 6, 0), (12, 3, 33, 5, 1), (12, 3, 30, 33, 2), (8, 3, 25, 7, 0),
                                               (8, 3, 30, 4, 2), (12, 2, 41, 6, 0), (12, 2, 40, 34, 1), (8, 2, 30, 5, 0),
                                               (8, 2, 31, 3, 1)])
def test_every_control_count_up_to_four_on_the_tensor_core_kernel(handle, oracle_mod, n, m, N, batch, mid_p, hess):
    """m = 2, 3 at n = 8, 12: knot records of odd length (the bulk copies start / end on the even doubles around
    them) — every m <= 4 is on the warp-per-instance kernel, not on the cooperative fallback."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=13 * n + 3 * m + mid_p, mid_p=mid_p, hess_mode=hess)
    _check(prob, handle, oracle_mod, truth_instances=(0, batch - 1))
    assert handle.last_kernel.startswith(f"kkt_wp_dmma<{n},{m},p={n}/{mid_p}/{n}"), handle.last_kernel


@pytest.mark.parametrize("hess,soc", [(1, False), (2, False), (1, True)])
@pytest.mark.parametrize("n,m,N,batch,mid_p", [(64, 16, 12, 3, 1), (64, 16, 13, 2, 2), (64, 16, 30, 2, 3), (48, 16, 12, 3, 1),
                                               (32, 8, 14, 3, 1), (32, 8, 15, 2, 4), (24, 8, 21, 4, 3), (16, 8, 20, 5, 1),
                                               (16, 8, 21, 3, 2), (16, 8, 30, 2, 4)])
def test_stage_constraints_on_the_cta_kernels(handle, oracle_mod, n, m, N, batch, mid_p, hess, soc):
    """Mid-horizon stage constraints (p = [n, ps, ..., ps, n], test/problems.jl:39-43) at the large-state sizes stay on the
    CTA-per-instance tensor-core kernels: ps <= 4 rows per knot as vector work beside the tile algebra.  Odd ps puts
    knot records on odd doubles (the pre-pass then stages [A B] with plain loads): batches > 1, both parities of N.
    Tolerance: 1e-10, or 4x the error the reference's own operation order (the oracle) makes on the input if larger."""
    from oracle import dense_kkt
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=7 * n + mid_p, mid_p=mid_p, hess_mode=hess)
    dz, lam, info, res = ops.kkt_solve_problem(prob, soc=soc, want_res=True, handle=handle)
    assert handle.last_kernel.startswith(f"kkt_cta_dmma<{n},{m},p={n}/{mid_p}/{n}"), handle.last_kernel
    dzo, lamo, infoo, reso = oracle_mod.kkt_solve(prob, soc=soc, want_res=True)
    assert (info == 0).all() and (infoo == 0).all()
    base = 1e-9 if soc else TOL
    for i in range(batch):
        zt, lt = dense_kkt.kkt_truth(prob, i, soc=soc)
        tol = max(base, 4.0 * max(_rel(dzo[i], zt), _rel(lamo[i], lt)))
        assert _rel(dz[i], zt) <= tol and _rel(lam[i], lt) <= tol, (i, tol, _rel(dz[i], zt), _rel(lam[i], lt))
        assert _rel(dz[i], dzo[i]) <= 2 * tol and _rel(lam[i], lamo[i]) <= 2 * tol
        assert np.linalg.norm(res[i] - reso[i]) <= 2 * tol * max(1.0, np.linalg.norm(reso[i]))
        rs, rp = dense_kkt.kkt_residuals(prob, i, dz[i], lam[i], soc=soc)
        assert rs <= 10 * base and rp <= 10 * base, (rs, rp)


def _per_knot_pattern(prob, seed, hi):
    """Keep a random number (0..hi) of the stage rows of every interior knot."""
    rng = np.random.default_rng(seed)
    p = prob["p"].copy()
    for k in range(1, prob["N"] - 1):
        p[k] = int(rng.integers(0, hi + 1))
        prob["C"][k] = prob["C"][k][:, :p[k]]
        prob["c"][k] = prob["c"][k][:, :p[k]]
    prob["p"] = p
    return prob


@pytest.mark.parametrize("hess,soc", [(1, False), (2, False), (0, False), (1, True)])
@pytest.mark.parametrize("n,m,N,batch,hi", [(12, 4, 40, 7, 3), (12, 4, 31, 33, 2), (8, 4, 30, 5, 3), (12, 3, 33, 6, 2),
                                            (8, 2, 30, 34, 1), (12, 2, 25, 3, 1)])
def test_per_knot_stage_rows_on_the_tensor_core_kernel(handle, oracle_mod, n, m, N, batch, hi, hess, soc):
    """The reference sizes every knot freely (src/conblocks.jl:74-96): a different number of stage rows on every
    interior knot (<= 4) stays on the warp-per-instance kernel; record and multiplier offsets come from the per-knot
    tables of the general path."""
    prob = _per_knot_pattern(problems.random_lqr_kkt(n, m, N, batch, seed=17 * n + hi, mid_p=hi, hess_mode=hess), N + hi, hi)
    assert len(set(prob["p"][1:-1].tolist())) > 1
    _check(prob, handle, oracle_mod, soc=soc, tol=1e-9 if soc else TOL, res_tol=1e-9 if soc else TOL,
           truth_instances=(0, batch - 1))
    assert handle.last_kernel.startswith(f"kkt_wp_dmma<{n},{m},p={n}/per-knot<={max(prob['p'][1:-1])}/{n}"), handle.last_kernel


def test_stage_constraints_match_cooperative_kernel_and_report_info(handle):
    prob = problems.random_lqr_kkt(12, 4, 50, 9, seed=4, mid_p=2, hess_mode=1)
    dz1, lam1, i1, r1 = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
    assert handle.last_kernel.startswith("kkt_wp_dmma<12,4,p=12/2/12")
    handle.set_option("kkt_variant", 2)
    try:
        dz2, lam2, i2, r2 = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
        assert handle.last_kernel.startswith("kkt_coop")
    finally:
        handle.set_option("kkt_variant", 0)
    assert (i1 == 0).all() and (i2 == 0).all()
    assert _rel(dz1, dz2) <= 1e-10 and _rel(lam1, lam2) <= 1e-10
    assert np.abs(r1 - r2).max() <= 1e-9 * max(1.0, np.abs(r2).max())
    # two identical stage rows at knot 7 of instance 3: the stage block B' is singular -> info names knot 8, stage 1
    prob["C"][7][3, 1] = prob["C"][7][3, 0]
    _, _, info = ops.kkt_solve_problem(prob, handle=handle)
    assert info[3] // 1000 == 8 and (info[3] % 1000) // 100 == 1 and (np.delete(info, 3) == 0).all(), info


def _free_final(prob):
    """Drop the goal rows: p_N = 0 (the MPC form: initial condition, dynamics, stage rows, free final state)."""
    prob["p"] = prob["p"].copy()
    prob["p"][-1] = 0
    b = prob["q"].shape[0]
    prob["C"][-1] = np.zeros((b, 0, prob["n"]))
    prob["c"][-1] = np.zeros((b, 0))
    return prob


@pytest.mark.parametrize("hess,soc", [(1, False), (2, False), (0, False), (1, True)])
@pytest.mark.parametrize("n,m,N,batch,mid_p,kern", [
    (12, 4, 30, 7, 0, "kkt_wp_dmma<12,4"), (12, 4, 31, 5, 2, "kkt_wp_dmma<12,4"), (8, 2, 20, 33, 1, "kkt_wp_dmma<8,2"),
    (4, 1, 25, 70, 0, "kkt_tpi<4,1,p=4/0/0"), (6, 3, 20, 33, 1, "kkt_tpi<6,3,p=6/1/0"), (3, 2, 41, 9, 0, "kkt_tpi<3,2,p=3/0/0"),
    (5, 2, 20, 6, 1, "kkt_tpi<5,2,p=5/1/0"), (6, 3, 20, 6, 2, "kkt_wp_dmma<8,4"), (10, 3, 25, 4, 0, "kkt_wp_dmma<12,4"),
    (14, 7, 12, 5, 1, "kkt_cta_dmma<16,8"), (64, 16, 9, 2, 0, "kkt_cta_dmma<64,16"), (24, 8, 12, 3, 2, "kkt_cta_dmma<24,8")])
def test_free_final_state_on_the_tuned_kernels(handle, oracle_mod, n, m, N, batch, mid_p, kern, hess, soc):
    """No goal rows (p_N = 0).  Small shapes have thread-per-instance instantiations of their own; above them the problem
    is embedded with a ZERO goal block and the tuned kernel leaves mu_N = 0 instead of inverting the last Schur block;
    the multiplier vector that comes back has no mu_N entries."""
    from oracle import dense_kkt
    prob = _free_final(problems.random_lqr_kkt(n, m, N, batch, seed=3 * n + m + mid_p, mid_p=mid_p, hess_mode=hess))
    dz, lam, info, res = ops.kkt_solve_problem(prob, soc=soc, want_res=True, handle=handle)
    if hess == 0 and n > 12:
        assert handle.last_kernel.startswith("kkt_coop")
    else:
        assert handle.last_kernel.startswith(kern), handle.last_kernel
        assert ("free final state padded" in handle.last_kernel) == (not kern.startswith("kkt_tpi")), handle.last_kernel
    dzo, lamo, infoo, reso = oracle_mod.kkt_solve(prob, soc=soc, want_res=True)
    assert (info == 0).all() and (infoo == 0).all() and lam.shape == lamo.shape
    base = 1e-9 if soc else TOL
    for i in range(batch):
        zt, lt = dense_kkt.kkt_truth(prob, i, soc=soc)
        tol = max(base, 4.0 * max(_rel(dzo[i], zt), _rel(lamo[i], lt)))
        assert _rel(dz[i], zt) <= tol and _rel(lam[i], lt) <= tol, (i, tol, _rel(dz[i], zt), _rel(lam[i], lt))
        assert np.linalg.norm(res[i] - reso[i]) <= 2 * tol * max(1.0, np.linalg.norm(reso[i]))


def test_free_final_state_resolve_of_ill_conditioned_instances(handle, oracle_mod):
    """The re-solve of flagged instances runs the general kernel on the problem as it is (no goal rows) inside the tuned
    kernel's padded layout (its own per-instance strides)."""
    from oracle import dense_kkt
    prob = _free_final(problems.random_lqr_kkt(12, 4, 30, 9, seed=8, mid_p=1, hess_mode=1))
    prob["Q"][::2] *= 1e3
    prob["R"][::2] *= 1e-3
    dz, lam, info = ops.kkt_solve_problem(prob, handle=handle)
    assert "+kkt_coop[" in handle.last_kernel and "free final state" in handle.last_kernel, handle.last_kernel
    dzo, lamo, infoo = oracle_mod.kkt_solve(prob)
    assert (info == 0).all() and (infoo == 0).all()
    for i in range(9):
        zt, lt = dense_kkt.kkt_truth(prob, i)
        tol = max(TOL, 4.0 * max(_rel(dzo[i], zt), _rel(lamo[i], lt)))
        assert _rel(dz[i], zt) <= tol and _rel(lam[i], lt) <= tol, (i, tol)
