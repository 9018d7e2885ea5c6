"""The gains-gradient oracle (oracle/riccati_gain_grad.py) against complex-step derivatives of a complex128
restatement of the Riccati recursion, element by element for every input (CPU only)."""
import numpy as np
import pytest

from oracle.riccati_gain_grad import gain_grad, riccati_total_grad
from oracle.riccati_grad import riccati_grad
from lqr_b200 import problems

ARGS = ("A", "B", "Q", "R", "q", "r", "Qf", "qf")
SYMMETRIC = ("Q", "R", "Qf")
H = 1e-30


def _gains_complex(prob):
    """K (b, N-1, m, n), kff (b, N-1, m) of the recursion in complex128 (no symmetrisation needed: the perturbed
    matrices stay symmetric)"""
    n, m, N = prob["n"], prob["m"], prob["N"]
    lti = bool(prob.get("lti", False))
    b = prob["Qf"].shape[0]

    def at(s, k, shape):
        a = prob.get(s)
        if a is None:
            return np.zeros((b,) + shape)
        return a if lti else a[:, k]
    P, p = prob["Qf"], (np.zeros((b, n)) if prob.get("qf") is None else prob["qf"])
    K = np.zeros((b, N - 1, m, n), complex)
    kff = np.zeros((b, N - 1, m), complex)
    for k in range(N - 2, -1, -1):
        A, B, Q, R = (at(s, k, ()) for s in ("A", "B", "Q", "R"))
        q, r = at("q", k, (n,)), at("r", k, (m,))
        Bt = np.swapaxes(B, -1, -2)
        G, Hm, h = R + Bt @ P @ B, Bt @ P @ A, r + np.einsum("bji,bj->bi", B, p)
        Kf = np.linalg.solve(G, np.concatenate([Hm, h[:, :, None]], axis=2))
        K[:, k], kff[:, k] = Kf[:, :, :n], Kf[:, :, n]
        P = Q + np.swapaxes(A, -1, -2) @ P @ A - np.swapaxes(Hm, -1, -2) @ K[:, k]
        p = q + np.einsum("bji,bj->bi", A, p) - np.einsum("bji,bj->bi", K[:, k], h)
    return K, kff


def _complex_step(prob, dK, dkff):
    """d/dt of l = sum(dK * K) + sum(dkff * kff) along every element of every input of instance 0 (a symmetric matrix
    at (i, j) and (j, i) together), all perturbed copies evaluated as one batch"""
    present = [k for k in ARGS if prob.get(k) is not None]
    base = {k: np.asarray(prob[k])[:1] for k in present}
    dirs = []
    for k in present:
        shape = base[k].shape[1:]
        for idx in np.ndindex(*shape):
            if k in SYMMETRIC and idx[-2] > idx[-1]:
                continue
            E = np.zeros(shape)
            E[idx] = 1.0
            if k in SYMMETRIC:
                E[idx[:-2] + (idx[-1], idx[-2])] = 1.0
            dirs.append((k, idx, E))
    batch = {k: np.repeat(base[k].astype(complex), len(dirs), axis=0) for k in present}
    for d, (k, _, E) in enumerate(dirs):
        batch[k][d] += 1j * H * E
    K, kff = _gains_complex(dict(prob, **batch))
    loss = np.zeros(len(dirs), complex)
    if dK is not None:
        loss += (K * dK[:1]).reshape(len(dirs), -1).sum(axis=1)
    if dkff is not None:
        loss += (kff * dkff[:1]).reshape(len(dirs), -1).sum(axis=1)
    return [(k, idx, loss[d].imag / H) for d, (k, idx, _) in enumerate(dirs)]


CASES = [  # (n, m, N, lti, affine, cotangents)
    (3, 2, 5, False, True, "both"), (3, 2, 5, True, True, "both"), (4, 1, 6, False, True, "both"),
    (4, 1, 6, True, False, "both"), (3, 2, 5, False, False, "K"), (3, 2, 5, False, True, "kff"),
    (5, 3, 4, True, True, "K"), (4, 1, 6, False, True, "kff"),
]


@pytest.mark.parametrize("n,m,N,lti,affine,cot", CASES)
def test_gain_oracle_matches_complex_step(n, m, N, lti, affine, cot):
    prob = problems.random_lqr_riccati(n, m, N, 2, seed=n * 10 + m + lti, dt=0.1, lti=lti)
    if not affine:
        prob.update(q=None, r=None, qf=None)
    rng = np.random.default_rng(n + m)
    dK = rng.standard_normal((2, N - 1, m, n)) if cot in ("K", "both") else None
    dkff = rng.standard_normal((2, N - 1, m)) if cot in ("kff", "both") else None
    g = gain_grad(prob, dK, dkff)
    seen = set()
    for k, idx, cs in _complex_step(prob, dK, dkff):
        an = g[k][(0,) + idx]
        if k in SYMMETRIC and idx[-2] != idx[-1]:
            an = an + g[k][(0,) + idx[:-2] + (idx[-1], idx[-2])]
        scale = max(np.abs(g[k][0]).max(), 1e-300)
        assert abs(an - cs) <= 1e-12 * scale, (k, idx, an, cs)
        seen.add(k)
    assert seen == {k for k in ARGS if prob.get(k) is not None}
    assert not g["x0"].any()
    for k in SYMMETRIC:
        np.testing.assert_allclose(g[k], np.swapaxes(g[k], -1, -2), rtol=0, atol=1e-14 * np.abs(g[k]).max())


def test_total_oracle_is_the_z_part_plus_the_gains_part():
    n, m, N = 4, 2, 6
    prob = problems.random_lqr_riccati(n, m, N, 3, seed=5, dt=0.1)
    rng = np.random.default_rng(0)
    dZ = rng.standard_normal((3, N * n + (N - 1) * m))
    dK, dkff = rng.standard_normal((3, N - 1, m, n)), rng.standard_normal((3, N - 1, m))
    tot, gz, gg = riccati_total_grad(prob, dZ, dK, dkff), riccati_grad(prob, dZ), gain_grad(prob, dK, dkff)
    for k in tot:
        np.testing.assert_array_equal(tot[k], gz[k] + gg[k])
    only = riccati_total_grad(prob, None, dK, None)
    for k, v in gain_grad(prob, dK, None).items():
        np.testing.assert_array_equal(only[k], v)
