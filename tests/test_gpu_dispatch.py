"""GPU: which kernel family runs for a shape and the options, for both solvers (the KKT and the Riccati routing
tables), and the conditioning record of a KKT call whose tuned-kernel work is split into chunks."""
import numpy as np
import pytest

from lqr_b200 import _lib, ops, problems

pytestmark = pytest.mark.gpu


def _problem(n, m, N, mid_p=0, hess=1, form=""):
    """A batch of 3 well-conditioned problems.  form: "free" drops the goal rows (p_N = 0), "waypoint" keeps the stage
    rows on one interior knot only, "d2" passes an explicit D2."""
    prob = problems.random_lqr_kkt(n, m, N, 3, seed=n + m + N, mid_p=mid_p, hess_mode=hess, explicit_D2=form == "d2")
    if form == "free":
        prob["p"] = prob["p"].copy()
        prob["p"][-1] = 0
        prob["C"][-1] = np.zeros((3, 0, n))
        prob["c"][-1] = np.zeros((3, 0))
    if form == "waypoint":
        prob["p"] = prob["p"].copy()
        for k in range(1, N - 1):
            if k != N // 2:
                prob["p"][k] = 0
                prob["C"][k] = np.zeros((3, 0, n + m))
                prob["c"][k] = np.zeros((3, 0))
    return prob


def _solve_packed(handle, prob, misaligned):
    """pack -> solve_packed -> unpack on device buffers; `misaligned` puts the packed data 8 bytes off 16-byte
    alignment."""
    import torch
    f = ops.kkt_flatten(prob)
    n, m, N, b, p, hm = f["n"], f["m"], f["N"], f["batch"], f["p"], f["hess_mode"]
    NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
    ldb = _lib.padded_batch(b)
    names = ("Q", "R", "Hux", "q", "r", "A", "B", "d", "D2", "C", "c")
    dev = {k: (None if f[k] is None else torch.from_numpy(np.ascontiguousarray(f[k])).cuda()) for k in names}
    z = lambda r: torch.zeros(ldb * r, dtype=torch.float64, device="cuda")  # noqa: E731
    base = z(_lib.kkt_data_rows(n, m, N, p, hm) + 1)
    data = base[1:] if misaligned else base
    assert data.data_ptr() % 16 == (8 if misaligned else 0)
    dzp, mp = z(NN), z(P)
    dz = torch.zeros(b, NN, dtype=torch.float64, device="cuda")
    mult = torch.zeros(b, P, dtype=torch.float64, device="cuda")
    info = torch.zeros(b, dtype=torch.int32, device="cuda")
    handle.set_stream(torch.cuda.current_stream().cuda_stream)
    try:
        ops.kkt_pack(handle, n, m, N, b, p, hm, *[dev[k] for k in names], data)
        ops.kkt_solve_packed(handle, n, m, N, b, p, hm, False, 0, data, dzp, mp, None, info)
        ops.kkt_unpack(handle, n, m, N, b, p, hm, False, dzp, mp, None, dz, mult)
        torch.cuda.synchronize()
    finally:
        handle.set_stream(None)
    return dz.cpu().numpy(), mult.cpu().numpy(), info.cpu().numpy()


# (problem, options, call) -> the kernel name the call reports.  call: "host" = lqrb_kkt_solve_f64 on host buffers,
# "packed" / "misaligned" = lqrb_kkt_solve_packed_f64 with 16-byte aligned / misaligned packed data.
ROUTES = [
    # every family on its own shapes
    (dict(n=4, m=1, N=12), {}, "host", "kkt_tpi<4,1,p=4/0/4,hess=1>"),
    (dict(n=6, m=3, N=12, mid_p=1, hess=0), {}, "host", "kkt_tpi<6,3,p=6/1/6,hess=0>"),
    (dict(n=4, m=1, N=12, form="free"), {}, "host", "kkt_tpi<4,1,p=4/0/0,hess=1>"),
    (dict(n=12, m=4, N=12), {}, "host", "kkt_hw<12,4,p=12/0/12,hess=1>"),
    (dict(n=8, m=4, N=12, hess=2), {}, "host", "kkt_hw<8,4,p=8/0/8,hess=2>"),
    (dict(n=12, m=3, N=12), {}, "host", "kkt_wp_dmma<12,3,p=12/0/12,hess=1>"),
    (dict(n=8, m=2, N=20, mid_p=1, hess=2), {}, "host", "kkt_wp_dmma<8,2,p=8/1/8,hess=2>"),
    (dict(n=64, m=16, N=6), {}, "host", "kkt_cta_dmma<64,16,p=64/0/64,hess=1>"),
    (dict(n=16, m=8, N=8, mid_p=1, hess=2), {}, "host", "kkt_cta_dmma<16,8,p=16/1/16,hess=2>"),
    # dense Hessian at n = 12 and above it
    (dict(n=12, m=4, N=12, mid_p=1, hess=0), {}, "host", "kkt_wp_dmma<12,4,p=12/1/12,hess=0>"),
    (dict(n=16, m=8, N=8, hess=0), {}, "host", "kkt_coop<G=32>(n=16,m=8,smem-ws)"),
    (dict(n=14, m=7, N=8, hess=0), {}, "host", "kkt_coop<G=32>(n=14,m=7,smem-ws)"),
    # irregular stage rows, more than 4 stage rows, explicit D2
    (dict(n=12, m=4, N=12, mid_p=2, form="waypoint"), {}, "host", "kkt_wp_dmma<12,4,p=12/per-knot<=2/12,hess=1>"),
    (dict(n=12, m=4, N=10, mid_p=5, form="waypoint"), {}, "host", "kkt_coop<G=32>(n=12,m=4,smem-ws)"),
    (dict(n=16, m=8, N=10, mid_p=5), {}, "host", "kkt_coop<G=32>(n=16,m=8,smem-ws)"),
    (dict(n=12, m=4, N=10, form="d2"), {}, "host", "kkt_coop<G=32>(n=12,m=4,smem-ws)"),
    (dict(n=4, m=1, N=10, form="d2"), {}, "host", "kkt_coop<G=4>(n=4,m=1,smem-ws)"),
    (dict(n=16, m=8, N=8, form="d2"), {}, "host", "kkt_coop<G=32>(n=16,m=8,smem-ws)"),
    # padding into each class
    (dict(n=10, m=3, N=12), {}, "host", "kkt_hw<12,4,p=12/0/12,hess=1>+kkt_coop[3 ill-conditioned] <- (10,3) padded"),
    (dict(n=7, m=2, N=12, mid_p=1), {}, "host", "kkt_wp_dmma<8,3,p=8/1/8,hess=1>+kkt_coop[1 ill-conditioned] <- (7,2) padded"),
    (dict(n=10, m=3, N=12, hess=0), {}, "host", "kkt_wp_dmma<12,4,p=12/0/12,hess=0>+kkt_coop[3 ill-conditioned] <- (10,3) padded"),
    (dict(n=14, m=7, N=8), {}, "host", "kkt_cta_dmma<16,8,p=16/0/16,hess=1>+kkt_coop[3 ill-conditioned] <- (14,7) padded"),
    (dict(n=40, m=12, N=6, mid_p=1, hess=2), {}, "host", "kkt_cta_dmma<48,16,p=48/1/48,hess=2>+kkt_coop[3 ill-conditioned] <- (40,12) padded"),
    (dict(n=10, m=3, N=12, form="free"), {}, "host", "kkt_wp_dmma<12,4,p=12/0/12,hess=1> <- (10,3) free final state padded"),
    (dict(n=12, m=4, N=12, form="free"), {}, "host", "kkt_wp_dmma<12,4,p=12/0/12,hess=1> <- (12,4) free final state padded"),
    (dict(n=14, m=7, N=8, form="free"), {}, "host", "kkt_cta_dmma<16,8,p=16/0/16,hess=1> <- (14,7) free final state padded"),
    (dict(n=4, m=1, N=16, mid_p=1, form="waypoint"), {}, "host", "kkt_wp_dmma<8,2,p=8/per-knot<=1/8,hess=1> <- (4,1) padded"),
    (dict(n=14, m=7, N=10, mid_p=5), {}, "host", "kkt_coop<G=32>(n=14,m=7,smem-ws)"),
    # kkt_variant = 2: the cooperative kernel everywhere
    (dict(n=4, m=1, N=12), {"kkt_variant": 2}, "host", "kkt_coop<G=4>(n=4,m=1,smem-ws)"),
    (dict(n=12, m=4, N=12), {"kkt_variant": 2}, "host", "kkt_coop<G=32>(n=12,m=4,smem-ws)"),
    (dict(n=12, m=3, N=12), {"kkt_variant": 2}, "host", "kkt_coop<G=32>(n=12,m=3,smem-ws)"),
    (dict(n=64, m=16, N=6), {"kkt_variant": 2}, "host", "kkt_coop<G=256>(n=64,m=16,gmem-ws)"),
    (dict(n=10, m=3, N=12), {"kkt_variant": 2}, "host", "kkt_coop<G=16>(n=10,m=3,smem-ws)"),
    # kkt_variant = 5: the warp-per-instance kernel where the half-warp kernel also has the shape
    (dict(n=12, m=4, N=12), {"kkt_variant": 5}, "host", "kkt_wp_dmma<12,4,p=12/0/12,hess=1>"),
    (dict(n=8, m=4, N=12, hess=2), {"kkt_variant": 5}, "host", "kkt_wp_dmma<8,4,p=8/0/8,hess=2>"),
    (dict(n=12, m=3, N=12), {"kkt_variant": 5}, "host", "kkt_wp_dmma<12,3,p=12/0/12,hess=1>"),
    (dict(n=10, m=3, N=12), {"kkt_variant": 5}, "host", "kkt_wp_dmma<12,4,p=12/0/12,hess=1>+kkt_coop[3 ill-conditioned] <- (10,3) padded"),
    (dict(n=64, m=16, N=6), {"kkt_variant": 5}, "host", "kkt_cta_dmma<64,16,p=64/0/64,hess=1>"),
    (dict(n=4, m=1, N=12), {"kkt_variant": 5}, "host", "kkt_tpi<4,1,p=4/0/4,hess=1>"),
    # kkt_pad = 0
    (dict(n=10, m=3, N=12), {"kkt_pad": 0}, "host", "kkt_coop<G=16>(n=10,m=3,smem-ws)"),
    (dict(n=14, m=7, N=8), {"kkt_pad": 0}, "host", "kkt_coop<G=32>(n=14,m=7,smem-ws)"),
    (dict(n=10, m=3, N=12, form="free"), {"kkt_pad": 0}, "host", "kkt_coop<G=16>(n=10,m=3,smem-ws)"),
    (dict(n=12, m=4, N=12), {"kkt_pad": 0}, "host", "kkt_hw<12,4,p=12/0/12,hess=1>"),
    (dict(n=10, m=3, N=12), {"kkt_pad": 0, "kkt_variant": 5}, "host", "kkt_coop<G=16>(n=10,m=3,smem-ws)"),
    # the packed entry point, with aligned and misaligned data
    (dict(n=12, m=4, N=12), {}, "packed", "kkt_hw<12,4,p=12/0/12,hess=1>"),
    (dict(n=10, m=3, N=12), {}, "packed", "kkt_hw<12,4,p=12/0/12,hess=1>+kkt_coop[3 ill-conditioned] <- (10,3) padded"),
    (dict(n=4, m=1, N=12), {}, "misaligned", "kkt_tpi<4,1,p=4/0/4,hess=1>"),
    (dict(n=12, m=4, N=12), {}, "misaligned", "kkt_coop<G=32>(n=12,m=4,smem-ws)"),
    (dict(n=12, m=3, N=12), {}, "misaligned", "kkt_coop<G=32>(n=12,m=3,smem-ws)"),
    (dict(n=64, m=16, N=6), {}, "misaligned", "kkt_coop<G=256>(n=64,m=16,gmem-ws)"),
    (dict(n=10, m=3, N=12), {}, "misaligned", "kkt_coop<G=16>(n=10,m=3,smem-ws)"),
]

_DEFAULTS = {"kkt_variant": 0, "kkt_pad": 1}


def _route(handle, shape, opts, call):
    prob = _problem(**shape)
    for k, v in opts.items():
        handle.set_option(k, v)
    try:
        if call == "host":
            dz, lam, info = ops.kkt_solve_problem(prob, handle=handle)
        else:
            dz, lam, info = _solve_packed(handle, prob, call == "misaligned")
    finally:
        for k in opts:
            handle.set_option(k, _DEFAULTS[k])
    return handle.last_kernel, prob, dz, lam, info


@pytest.mark.parametrize("shape,opts,call,kern", ROUTES)
def test_route(handle, oracle_mod, shape, opts, call, kern):
    name, prob, dz, lam, info = _route(handle, shape, opts, call)
    assert name == kern
    dzo, lamo, infoo = oracle_mod.kkt_solve(prob)
    assert (info == 0).all() and (infoo == 0).all()
    assert np.linalg.norm(dz - dzo) <= 1e-9 * np.linalg.norm(dzo) and np.linalg.norm(lam - lamo) <= 1e-9 * np.linalg.norm(lamo)


def _riccati_solve_packed(handle, prob, misaligned):
    """riccati_pack -> riccati_solve_packed -> riccati_unpack on device buffers; `misaligned` puts the packed knots 8
    bytes off 16-byte alignment."""
    import torch
    f = ops.riccati_flatten(prob)
    n, m, N, b = f["n"], f["m"], f["N"], f["batch"]
    flags = _lib.FLAG_LTI if f["lti"] else 0
    L = _lib.riccati_layout(n, m, N, flags)
    ldb = _lib.padded_batch(b)
    names = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")
    dev = {k: torch.from_numpy(f[k]).cuda() for k in names}
    z = lambda *s: torch.zeros(*s, dtype=torch.float64, device="cuda")  # noqa: E731
    base = z(ldb * L.knot_count * L.rows_per_knot + 1)
    knots = base[1:] if misaligned else base[:-1]
    assert knots.data_ptr() % 16 == (8 if misaligned else 0)
    term, Zp, gains = z(ldb * L.term_rows), z(ldb * L.z_rows), z(ldb * L.gain_rows)
    Z, K, kff = z(b, L.z_rows), z(b, N - 1, n, m), z(b, N - 1, m)
    info = torch.zeros(b, dtype=torch.int32, device="cuda")
    handle.set_stream(torch.cuda.current_stream().cuda_stream)
    try:
        ops.riccati_pack(handle, n, m, N, b, flags, *[dev[k] for k in names], knots, term)
        ops.riccati_solve_packed(handle, n, m, N, b, flags, knots, term, Zp, gains, info)
        ops.riccati_unpack(handle, n, m, N, b, Zp, gains, Z, K, kff)
        torch.cuda.synchronize()
    finally:
        handle.set_stream(None)
    X, U = ops.split_primals(Z.cpu().numpy(), n, m, N)
    return X, U, np.swapaxes(K.cpu().numpy(), -1, -2), kff.cpu().numpy(), info.cpu().numpy()


# (shape, options, call) -> the kernel name the call reports.  call: "host" = lqrb_riccati_f64 on host buffers,
# "packed" / "misaligned" = lqrb_riccati_solve_packed_f64 with 16-byte aligned / misaligned packed knots.
RICCATI_ROUTES = [
    # every family on its own shapes
    (dict(n=4, m=1, N=30), {}, "host", "riccati_tpi<4,1>[64x8]"),
    (dict(n=6, m=3, N=30), {}, "host", "riccati_tpi<6,3>[128x1]"),
    (dict(n=4, m=1, N=30, lti=True), {}, "host", "riccati_tpi<4,1>[lti][64x8]"),
    (dict(n=8, m=1, N=30), {}, "host", "riccati_dmma<8,1>"),
    (dict(n=12, m=4, N=30), {}, "host", "riccati_dmma<12,4>"),
    (dict(n=12, m=4, N=30, lti=True), {}, "host", "riccati_dmma<12,4>[lti]"),
    (dict(n=16, m=16, N=12), {}, "host", "riccati_cta_dmma<16,16>"),
    (dict(n=64, m=16, N=8), {}, "host", "riccati_cta_dmma<64,16>"),
    # padding into each class
    (dict(n=7, m=2, N=30), {}, "host", "riccati_dmma<8,2> <- (7,2) padded"),
    (dict(n=5, m=4, N=30), {}, "host", "riccati_dmma<8,4> <- (5,4) padded"),
    (dict(n=10, m=3, N=30), {}, "host", "riccati_dmma<12,3> <- (10,3) padded"),
    (dict(n=7, m=7, N=20), {}, "host", "riccati_cta_dmma<16,8> <- (7,7) padded"),
    (dict(n=13, m=2, N=20), {}, "host", "riccati_cta_dmma<16,8> <- (13,2) padded"),
    (dict(n=40, m=12, N=8), {}, "host", "riccati_cta_dmma<48,16> <- (40,12) padded"),
    # no padding target
    (dict(n=65, m=16, N=6), {}, "host", "riccati_coop<G=256>(n=65,m=16)"),
    # riccati_pad = 0
    (dict(n=10, m=3, N=30), {"riccati_pad": 0}, "host", "riccati_coop<G=32>(n=10,m=3)"),
    (dict(n=12, m=4, N=30), {"riccati_pad": 0}, "host", "riccati_dmma<12,4>"),
    # riccati_variant = 2: the cooperative kernel everywhere; other values act as 0
    (dict(n=4, m=1, N=30), {"riccati_variant": 2}, "host", "riccati_coop<G=32>(n=4,m=1)"),
    (dict(n=12, m=4, N=30), {"riccati_variant": 2}, "host", "riccati_coop<G=32>(n=12,m=4)"),
    (dict(n=64, m=16, N=8), {"riccati_variant": 2}, "host", "riccati_coop<G=256>(n=64,m=16)"),
    (dict(n=10, m=3, N=30), {"riccati_variant": 2}, "host", "riccati_coop<G=32>(n=10,m=3)"),
    (dict(n=10, m=3, N=30), {"riccati_variant": 1}, "host", "riccati_dmma<12,3> <- (10,3) padded"),
    # the packed entry point, with aligned and misaligned data
    (dict(n=4, m=1, N=30), {}, "misaligned", "riccati_tpi<4,1>[64x8]"),
    (dict(n=12, m=4, N=30), {}, "misaligned", "riccati_coop<G=32>(n=12,m=4)"),
    (dict(n=64, m=16, N=8), {}, "misaligned", "riccati_coop<G=256>(n=64,m=16)"),
    (dict(n=10, m=3, N=30), {}, "misaligned", "riccati_coop<G=32>(n=10,m=3)"),
    (dict(n=10, m=3, N=30), {}, "packed", "riccati_dmma<12,3> <- (10,3) padded"),
]

_RICCATI_DEFAULTS = {"riccati_variant": 0, "riccati_pad": 1}


@pytest.mark.parametrize("shape,opts,call,kern", RICCATI_ROUTES)
def test_riccati_route(handle, oracle_mod, shape, opts, call, kern):
    n, m, N = shape["n"], shape["m"], shape["N"]
    prob = problems.random_lqr_riccati(n, m, N, 3, seed=n + m + N, lti=shape.get("lti", False))
    for k, v in opts.items():
        handle.set_option(k, v)
    try:
        if call == "host":
            out = ops.riccati_solve_problem(prob, handle=handle)
        else:
            out = _riccati_solve_packed(handle, prob, call == "misaligned")
    finally:
        for k in opts:
            handle.set_option(k, _RICCATI_DEFAULTS[k])
    assert handle.last_kernel == kern
    ref = oracle_mod.riccati(prob)
    assert (out[4] == 0).all() and (ref[4] == 0).all()
    for got, want in zip(out[:4], ref[:4]):  # X, U, K, kff
        assert np.linalg.norm(got - want) <= 1e-9 * np.linalg.norm(want)


@pytest.mark.parametrize("b,opts", [(3600, {"scratch_budget_mb": 8}), (70, {"host_chunk": 32})])
def test_condition_record_covers_the_whole_call(handle, b, opts):
    """A (12, 4) problem on the half-warp kernel with every other instance's costs rescaled, so that each chunk has
    instances re-solved by the Cholesky-based kernel.  A small scratch budget splits the batch into chunks of one
    resident wave (3,552 instances on a 148-SM B200); host buffers are processed in chunks of `host_chunk`.  The conditioning record, the re-solve count and
    the kernel name describe the whole call, as for the same call in one chunk."""
    prob = problems.random_lqr_kkt(12, 4, 10, b, seed=41, mid_p=0, hess_mode=1)
    prob["Q"][::2] *= 1e3
    prob["R"][::2] *= 1e-3

    def run(**o):
        for k, v in o.items():
            handle.set_option(k, v)
        try:
            ops.kkt_solve_problem(prob, handle=handle)
        finally:
            handle.set_option("scratch_budget_mb", 49152)
            handle.set_option("host_chunk", 0)
        return handle.kkt_last_condition(b) + (handle.last_kernel,)

    bits0, resolved0, name0 = run()
    bits, resolved, name = run(**opts)
    assert name0.startswith("kkt_hw<12,4") and "+kkt_coop[" in name0
    assert (bits0 >= 0).all() and resolved0 == int((bits0 >= 6).sum()) > 0
    assert np.array_equal(bits, bits0) and resolved == resolved0 and name == name0, (resolved, resolved0, name, name0)
