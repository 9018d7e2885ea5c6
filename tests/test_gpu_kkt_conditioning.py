"""GPU: every KKT kernel family on ill-conditioned Hessian, actuator and stage-row blocks, against the extended-precision
global KKT solve (oracle/dense_kkt.py), and the info codes of every family against the C oracle.

The tuned kernels (kkt_hw2, kkt_wp, kkt_cta) form explicit inverses of H_k, Sigma_k and the stage block B' by
Gauss-Jordan without pivoting, where the reference factors them (src/cholesky_solve.jl:47-67).  Instances whose
conditioning estimate reaches `kkt_cond_bits` are solved again by the Cholesky-based kkt_coop.  The generators the other
KKT tests use keep every block well conditioned, so these inputs are built here:
  * the cost rescalings of test_gpu_conditioning.py;
  * near-parallel cheap actuators: B[..., j] = B[..., 0] + c B[..., j] for j >= 1 (c down to 1e-4) and R scaled by
    rs down to 1e-8 (m = 1: R x rs);
  * R = V diag(logspace) V' with an eigenvalue spread up to 1e12;
  * a dense Hessian close to indefinite: R - Hux Q^-1 Hux' keeps a fraction delta of R's smallest eigenvalue;
  * stage rows: two rows of one knot nearly parallel (c down to 1e-3), rows scaled over 10^+-4, and a row on knot 2
    whose state part is nearly orthogonal to range(B_1), so that only u_1 can satisfy it (x_1 is fixed by the initial
    rows).
Ill-conditioned and benign instances alternate in every batch.

Tolerance, per instance: the relative error of dz and of the multipliers against the truth must be
<= max(1e-10, 4 x the error of the C oracle, which runs the reference's operation order, on the same instance) — the
rule of test_gpu_conditioning.py.  tests/test_oracle.py checks the truth on these inputs against a 40-digit solve.

The info tests fix the code the header promises, (knot + 1) * 1000 + stage * 100 + pivot in the caller's z numbering,
for every family: each case must return exactly the C oracle's code."""
import contextlib

import numpy as np
import pytest

from lqr_b200 import ops, problems
from tests.test_gpu_conditioning import SCALES

pytestmark = pytest.mark.gpu

COND_BITS = 6  # the default of the kkt_cond_bits option

# (n, m, N, stage rows per interior knot, Hessian mode, form, expected kernel-name prefix, options, padded, tuned)
#   form "perknot": the stage rows sit on knots 2 and N/2 + 1 only
FAMILIES = [
    (4, 1, 16, 0, 1, "", "kkt_tpi<4,1,", {}, False, False),
    (6, 3, 16, 1, 0, "", "kkt_tpi<6,3,", {}, False, False),
    (12, 4, 20, 0, 1, "", "kkt_hw<12,4,", {}, False, True),
    (8, 4, 20, 0, 2, "", "kkt_hw<8,4,", {}, False, True),
    (12, 4, 20, 0, 1, "", "kkt_wp_dmma<12,4,", {"kkt_variant": 5}, False, True),
    *[(n, m, 20, 0, 1, "", f"kkt_wp_dmma<{n},{m},", {}, False, True) for n in (8, 12) for m in (1, 2, 3)],
    (12, 4, 20, 0, 0, "", "kkt_wp_dmma<12,4,", {}, False, True),
    (8, 2, 20, 0, 0, "", "kkt_wp_dmma<8,2,", {}, False, True),
    (12, 4, 20, 2, 1, "", "kkt_wp_dmma<12,4,", {}, False, True),
    (8, 4, 20, 3, 1, "", "kkt_wp_dmma<8,4,", {}, False, True),
    (12, 4, 20, 2, 1, "perknot", "kkt_wp_dmma<12,4,p=12/per-knot<=2", {}, False, True),
    (64, 16, 8, 0, 1, "", "kkt_cta_dmma<64,16,", {}, False, True),
    (24, 8, 12, 0, 1, "", "kkt_cta_dmma<24,8,", {}, False, True),
    (16, 8, 12, 2, 1, "", "kkt_cta_dmma<16,8,", {}, False, True),
    (32, 8, 10, 4, 1, "", "kkt_cta_dmma<32,8,", {}, False, True),
    (10, 3, 20, 0, 1, "", "kkt_hw<12,4,", {}, True, True),
    (7, 2, 20, 1, 1, "", "kkt_wp_dmma<8,3,", {}, True, True),
    (14, 7, 12, 0, 1, "", "kkt_cta_dmma<16,8,", {}, True, True),
    (20, 6, 12, 2, 1, "", "kkt_cta_dmma<24,8,", {}, True, True),
    (12, 4, 20, 2, 1, "", "kkt_coop<", {"kkt_variant": 2}, False, False),
    (10, 3, 20, 1, 0, "", "kkt_coop<", {"kkt_pad": 0}, False, False),
]
FAMILY_IDS = [f"{f[6].rstrip(',')}-{f[0]}x{f[1]}-ps{f[3]}-h{f[4]}" + (f"-{f[5]}" if f[5] else "") +
              ("-padded" if f[8] else "") + ("-" + ",".join(f[7]) if f[7] else "") for f in FAMILIES]
DEFAULTS = {"kkt_variant": 0, "kkt_pad": 1, "kkt_refine": 1}

# c stops at 1e-4 and 1e-3: beyond, the refined solve no longer agrees with a 40-digit one (tests/test_oracle.py)
PARALLEL = [(c, rs) for c in (1e-2, 1e-3, 1e-4) for rs in (1e-4, 1e-6, 1e-8)]
CHEAP = [(None, rs) for rs in (1e-4, 1e-6, 1e-8)]  # m = 1: a cheap single actuator
SPREADS = [1e4, 1e8, 1e12]
DELTAS = [1e-2, 1e-4, 1e-6, 1e-8]
ROW_PARALLEL = [("parallel", c) for c in (1e-2, 1e-3)]
ROW_SCALED = [("scaled", e) for e in (2.0, 4.0)]
ROW_REACH = [("reach", eps) for eps in (1e-2, 1e-3)]


def kind_params(kind, m, mid_p, hess):
    """The ill-conditioned variants of an input kind that apply to a shape ([] where the kind does not apply)."""
    if kind == "scales":
        return list(SCALES)
    if kind == "parallel":
        return PARALLEL if m >= 2 else CHEAP
    if kind == "spread":
        return SPREADS if m >= 2 else []
    if kind == "dense":
        return DELTAS if hess == 0 else []
    if kind == "rows":
        return (ROW_PARALLEL if mid_p >= 2 else []) + (ROW_SCALED + ROW_REACH if mid_p >= 1 else [])
    raise ValueError(kind)


KINDS = ("scales", "parallel", "spread", "dense", "rows")
CASES = [(kind, *f) for f in FAMILIES for kind in KINDS if kind_params(kind, f[1], f[3], f[4])]
CASE_IDS = [f"{c[0]}-{i}" for c, i in zip(CASES, [FAMILY_IDS[FAMILIES.index(c[1:])] for c in CASES])]

# Known misses, measured on a B200 (instance: kernel error / C-oracle error).  Strict: a case that starts to pass must
# leave this list.  The Cholesky-based kkt_coop, which re-solves flagged instances, misses the 4x rule itself on some of
# them, so flagging more instances would not close these.
KNOWN_MISSES = {
    "scales-kkt_wp_dmma<12,4-12x4-ps2-h1": "instance 5 re-solved by kkt_coop: 5.7e-6 / 1.3e-6",
    "scales-kkt_wp_dmma<8,4-8x4-ps3-h1": "benign instance 12 flagged (2^6) by the Sigma estimate; accuracy passes",
    "rows-kkt_cta_dmma<32,8-32x8-ps4-h1": "weak row (1e-3), not flagged: 5.5e-6 / 1.1e-6",
    "parallel-kkt_cta_dmma<24,8-20x6-ps2-h1-padded": "instance 17 (c = 1e-4, rs = 1e-8) re-solved by kkt_coop: 1.9e-7 / 3.8e-8",
    "spread-kkt_cta_dmma<32,8-32x8-ps4-h1": "benign instance 2 with 4 random stage rows: 2.0e-10 / 5.1e-11",
    "rows-kkt_wp_dmma<8,3-7x2-ps1-h1-padded": "weak row (1e-2), not flagged: 3.3e-10 / 6.7e-11",
    "rows-kkt_coop<-10x3-ps1-h0-kkt_pad": "kkt_coop itself, weak row (1e-2): 8.5e-9 / 1.6e-9",
}
CASE_PARAMS = [pytest.param(*c, id=i, marks=[pytest.mark.xfail(strict=True, reason=KNOWN_MISSES[i])] if i in KNOWN_MISSES
                            else []) for c, i in zip(CASES, CASE_IDS)]


@contextlib.contextmanager
def _options(handle, opts):
    for k, v in opts.items():
        handle.set_option(k, v)
    try:
        yield
    finally:
        for k in opts:
            handle.set_option(k, DEFAULTS[k])


def _solve(handle, prob, kern, opts, padded):
    with _options(handle, opts):
        out = ops.kkt_solve_problem(prob, want_res=True, handle=handle)
    name = handle.last_kernel
    assert name.startswith(kern) and ("padded" in name) == padded, name
    return out, name


# ------------------------------------------------------------------ inputs
def make_problem(n, m, N, batch, seed, mid_p=0, hess=1, form=""):
    """random_lqr_kkt; form "perknot" keeps the stage rows on knots 2 and N/2 + 1 (indices 1 and N // 2) only."""
    prob = problems.random_lqr_kkt(n, m, N, batch, seed=seed, mid_p=mid_p, hess_mode=hess)
    if form == "perknot":
        prob["p"] = prob["p"].copy()
        for k in range(1, N - 1):
            if k not in (1, N // 2):
                prob["p"][k] = 0
                prob["C"][k] = np.zeros((batch, 0, n + m))
                prob["c"][k] = np.zeros((batch, 0))
    return prob


def _rotation(rng, m):
    V, _ = np.linalg.qr(rng.standard_normal((m, m)))
    return V


def _near_parallel(prob, i, c, rs):
    if c is not None:
        B = prob["B"][i]
        B[..., 1:] = B[..., :1] + c * B[..., 1:]
    prob["R"][i] *= rs


def _spread_R(prob, i, spread, rng):
    m = prob["m"]
    for k in range(prob["N"] - 1):
        V = _rotation(rng, m)
        R = V @ np.diag(np.logspace(0.0, -np.log10(spread), m)) @ V.T
        prob["R"][i, k] = 0.5 * (R + R.T)


def _near_indefinite_hessian(prob, i, delta, rng):
    """Hux = sqrt((1 - delta) lmin) v (Lq w)' with R v = lmin v, Q = Lq Lq', |w| = 1: then
    R - Hux Q^-1 Hux' = R - (1 - delta) lmin v v' has smallest eigenvalue delta lmin."""
    n = prob["n"]
    for k in range(prob["N"] - 1):
        lam, V = np.linalg.eigh(prob["R"][i, k])
        w = rng.standard_normal(n)
        w /= np.linalg.norm(w)
        Lq = np.linalg.cholesky(prob["Q"][i, k])
        prob["Hux"][i, k] = np.sqrt((1.0 - delta) * lam[0]) * np.outer(V[:, 0], Lq @ w)


def _interior_row_knots(prob):
    return [k for k in range(1, prob["N"] - 1) if prob["p"][k] > 0]


def _stage_rows(prob, i, what, par, rng):
    n = prob["n"]
    knots = _interior_row_knots(prob)
    if what == "parallel":  # C_j = C_0 + c C_j on every knot with stage rows
        for k in knots:
            C = prob["C"][k][i]
            C[1:] = C[:1] + par * C[1:]
    elif what == "scaled":  # row j of knot k scaled by 10^(+-par), alternating over rows and knots
        for k in knots:
            for j in range(prob["p"][k]):
                s = 10.0 ** (par * (-1) ** (j + k))
                prob["C"][k][i][j] *= s
                prob["c"][k][i][j] *= s
    else:  # a row on knot 2 (index 1) whose state part is nearly orthogonal to range(B_1): only u_1 can satisfy it
        B0 = prob["B"][i, 0]
        Qb, _ = np.linalg.qr(B0)
        v = rng.standard_normal(n)
        v -= Qb @ (Qb.T @ v)
        v /= np.linalg.norm(v)
        b = Qb @ rng.standard_normal(Qb.shape[1])
        row = np.zeros(prob["C"][1].shape[-1])
        row[:n] = v + par * b / np.linalg.norm(b)
        prob["C"][1][i][0] = row


def _congruent_Hux(prob, i, Q0, R0):
    """After Q_k, R_k of instance i changed from Q0, R0: Hux <- Lr Lr0^-1 Hux Lq0^-T Lq' (L: Cholesky factors), so that
    the dense H_k stays as far from indefinite as before (the Schur complements are congruent)."""
    for k in range(prob["N"] - 1):
        Lq0, Lq = np.linalg.cholesky(Q0[k]), np.linalg.cholesky(prob["Q"][i, k])
        Lr0, Lr = np.linalg.cholesky(R0[k]), np.linalg.cholesky(prob["R"][i, k])
        prob["Hux"][i, k] = Lr @ np.linalg.solve(Lr0, np.linalg.solve(Lq0, prob["Hux"][i, k].T).T) @ Lq.T


def make_batch(kind, n, m, N, mid_p, hess, form, seed):
    """A batch of 2 J + 1 instances: benign at even positions, the J ill-conditioned variants of `kind` at odd ones."""
    params = kind_params(kind, m, mid_p, hess)
    prob = make_problem(n, m, N, 2 * len(params) + 1, seed, mid_p, hess, form)
    rng = np.random.default_rng(seed)
    for j, par in enumerate(params):
        i = 2 * j + 1
        Q0, R0 = prob["Q"][i].copy(), prob["R"][i].copy()
        if kind == "scales":
            qs, rs = par
            prob["Q"][i] *= qs
            prob["R"][i] *= rs
        elif kind == "parallel":
            _near_parallel(prob, i, *par)
        elif kind == "spread":
            _spread_R(prob, i, par, rng)
        elif kind == "dense":
            _near_indefinite_hessian(prob, i, par, rng)
        else:
            _stage_rows(prob, i, *par, rng)
        if hess == 0 and kind != "dense":
            _congruent_Hux(prob, i, Q0, R0)
    return prob


def truth(prob):
    from oracle import dense_kkt
    return [dense_kkt.kkt_truth(prob, i) for i in range(prob["q"].shape[0])]


def errors(dz, mult, tr):
    rel = lambda a, b: np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)  # noqa: E731
    return np.array([max(rel(dz[i], zt), rel(mult[i], lt)) for i, (zt, lt) in enumerate(tr)])


# ------------------------------------------------------------------ accuracy
@pytest.mark.parametrize("kind,n,m,N,mid_p,hess,form,kern,opts,padded,tuned", CASE_PARAMS)
def test_ill_conditioned_blocks(handle, oracle_mod, kind, n, m, N, mid_p, hess, form, kern, opts, padded, tuned):
    prob = make_batch(kind, n, m, N, mid_p, hess, form, seed=2000 + 31 * n + 7 * m + mid_p + 3 * hess)
    b = prob["q"].shape[0]
    (dz, mult, info, _), name = _solve(handle, prob, kern, opts, padded)
    dzo, multo, infoo = oracle_mod.kkt_solve(prob)
    tr = truth(prob)
    assert all(np.isfinite(zt).all() and np.isfinite(lt).all() for zt, lt in tr)
    assert (infoo == 0).all() and (info == 0).all(), (infoo.tolist(), info.tolist())
    e, eo = errors(dz, mult, tr), errors(dzo, multo, tr)
    bad = np.flatnonzero(e > np.maximum(1e-10, 4.0 * eo))
    assert bad.size == 0, [(int(i), f"kernel {e[i]:.2e}", f"oracle {eo[i]:.2e}") for i in bad]
    if tuned:
        bits, resolved = handle.kkt_last_condition(b)
        assert resolved == int((bits >= COND_BITS).sum())
        assert ("+kkt_coop[" in name) == (resolved > 0), name
        if not padded:  # (a padded shape mixes the pad states' unit blocks into its estimate; see DESIGN §2)
            assert (bits[::2] < COND_BITS).all(), bits.tolist()


# ------------------------------------------------------------------ info codes
def _indefinite(m, j, rng):
    """A symmetric R = L D L' (L unit lower triangular) whose potrf pivots are D: the first non-positive one is j."""
    L = np.eye(m) + np.tril(0.3 * rng.standard_normal((m, m)), -1)
    d = rng.uniform(0.5, 2.0, m)
    d[j] = -0.5
    R = (L * d) @ L.T
    return 0.5 * (R + R.T)


def _indefinite_dense(prob, i, k, j, rng):
    """Dense H_k whose Schur complement R - Hux Q^-1 Hux' is indefinite at its pivot j: potrf fails at n + j + 1."""
    Q, Hux = prob["Q"][i, k], prob["Hux"][i, k]
    prob["R"][i, k] = _indefinite(prob["m"], j, rng) + Hux @ np.linalg.solve(Q, Hux.T)


def _info_batch(n, m, N, mid_p, hess, form):
    """The failure cases that apply to a shape, each on its own instance between clean ones.  Returns the problem."""
    rng = np.random.default_rng(n * 37 + m + mid_p)
    cases = []
    if hess != 2:  # the diagonal mode inverts the diagonal as it is (the reference checks no pivot there)
        cases += [("Q", k, j) for k in (0, N // 2, N - 1) for j in sorted({0, n // 2, n - 1})]
        cases += [("R", N // 2, j) for j in sorted({0, m - 1})]
    if hess == 0:
        cases += [("H", 3, j) for j in sorted({0, m - 1})]
    if mid_p >= 2:
        cases += [("zero-rows", None, None)]
    if mid_p >= 1:
        cases += [("zero-row", None, 1)]
    cases += [("C1", 0, j) for j in sorted({0, n // 2})]
    if hess != 2:
        cases += [("two", None, None), ("rescaled", None, None)]
    prob = make_problem(n, m, N, 2 * len(cases) + 1, 7 * n + m + 100 * mid_p, mid_p, hess, form)
    knots = _interior_row_knots(prob)
    for c, (what, k, j) in enumerate(cases):
        i = 2 * c + 1
        if what == "Q":
            prob["Q"][i, k] = _indefinite(n, j, rng)
        elif what == "R":
            prob["R"][i, k] = _indefinite(m, j, rng)
        elif what == "H":
            _indefinite_dense(prob, i, k, j, rng)
        elif what == "zero-rows":  # two identical stage rows (both zero): the Schur block is singular at pivot 1
            prob["C"][knots[-1]][i][:2] = 0.0
        elif what == "zero-row":  # a vanishing stage row: B' is singular at that row's pivot
            prob["C"][knots[0]][i][-1] = 0.0
        elif what == "C1":  # a rank-deficient initial block
            prob["C"][0][i][j] = 0.0
        elif what == "two":  # a Schur-block failure early and a Hessian failure late: the Hessian's code wins
            prob["C"][0][i][n - 1] = 0.0
            prob["R"][i, N - 3] = _indefinite(m, m - 1, rng)
        else:  # rescaled (and so re-solved on the tuned families) and indefinite R at an interior knot
            prob["Q"][i] *= 1e3
            prob["R"][i] *= 1e-3
            prob["R"][i, N // 2 + 1] = _indefinite(m, 0, rng) * 1e-3
    return prob


@pytest.mark.parametrize("n,m,N,mid_p,hess,form,kern,opts,padded,tuned", FAMILIES, ids=FAMILY_IDS)
def test_info_code_matches_the_oracle(handle, oracle_mod, n, m, N, mid_p, hess, form, kern, opts, padded, tuned):
    prob = _info_batch(n, m, N, mid_p, hess, form)
    want = oracle_mod.kkt_solve(prob)[2]
    assert (want[::2] == 0).all() and (want[1::2] != 0).all(), want.tolist()
    (_, _, info, _), _ = _solve(handle, prob, kern, opts, padded)
    assert np.array_equal(info, want), (info.tolist(), want.tolist())


@pytest.mark.parametrize("n,m,N,mid_p,hess,form,kern,opts,padded,tuned", FAMILIES, ids=FAMILY_IDS)
def test_nan_instance_is_isolated(handle, n, m, N, mid_p, hess, form, kern, opts, padded, tuned):
    """A NaN in one instance's R, and in another run in one stage row, is reported by that instance only and changes
    no bit of any other instance — also when other instances of the batch are re-solved (instances 0 and 4 have
    rescaled costs)."""
    prob = make_problem(n, m, N, 5, 13 * n + m, mid_p, hess, form)
    for i in (0, 4):
        prob["Q"][i] *= 1e3
        prob["R"][i] *= 1e-3
    clean, _ = _solve(handle, prob, kern, opts, padded)
    assert (clean[2] == 0).all()
    knot = _interior_row_knots(prob)[0] if mid_p else 0
    for where in ("R", "C"):
        dirty_prob = {k: (v.copy() if isinstance(v, np.ndarray) else [a.copy() for a in v] if isinstance(v, list) else v)
                      for k, v in prob.items()}
        if where == "R":
            dirty_prob["R"][2, N // 2, m - 1, m - 1] = np.nan
        else:
            dirty_prob["C"][knot][2][0, n // 2] = np.nan
        dirty, _ = _solve(handle, dirty_prob, kern, opts, padded)
        assert dirty[2][2] != 0 and (np.delete(dirty[2], 2) == 0).all(), (where, dirty[2].tolist())
        for a, c in zip((clean[0], clean[1], clean[3]), (dirty[0], dirty[1], dirty[3])):
            assert np.array_equal(np.delete(a, 2, axis=0), np.delete(c, 2, axis=0)), where
