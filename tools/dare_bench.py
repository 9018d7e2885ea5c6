#!/usr/bin/env python
"""Cost of the batched DARE (lqrb_dare_f64) and its gradient (lqrb_dare_grad_f64), device-resident, next to what they
replace: the first gain of an LTI lqrb_riccati_f64 horizon long enough that K_0 is within 1e-12 of K (N - 1 knots with
rho^(2(N-1)) <= 1e-12 for the batch's largest rho(A - BK); the K_0 error reached is recorded), and
lqrb_riccati_grad_gains_f64 of <dK, K_0> at that horizon.  Inputs are the stable draws of
problems.dare_lti_riccati from a seed whose closed loop has rho(A - BK) <= 0.95 (a few draws in 10^4 come within 1e-3
of 1, and the horizon the alternative needs grows as 1 / log(1 / rho)).  Per shape: call times from CUDA events (warm-up, then windows of at least
0.35 s, the best window kept), the distribution of the doubling steps, FLOPs counted from the shapes and the steps
taken, and their fraction of the FP64 DFMA peak measured in the same run (lqrb_fp64_peak_f64).  The card's name and
power limit are read in the same run.  Prints one JSON line (and writes it to --out when given)."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lqr_b200 import _lib, ops, problems  # noqa: E402
from oracle import dare as od  # noqa: E402

SHAPES = [(4, 1, 65536), (12, 4, 16384), (64, 16, 4096)]
WINDOW_S = 0.35


def dare_flops(n, m, steps):
    """per instance: each doubling step forms W = I + GH (2n^3), its LU (2n^3/3), W^-1 [A | G] (4n^3) and five n x n
    products (10n^3); before it G_0 = B R^-1 B' (n^2 m + n m^2 + m^3/3); after it PA, PB, R + B'PB, B'PA and the gain
    solve (2n^3 + 4n^2 m + 2n m^2 + m^3/3 + 2 m^2 n)"""
    step = 2 * n**3 + 2 * n**3 / 3 + 4 * n**3 + 10 * n**3
    return steps * step + (n * n * m + n * m * m + m**3 / 3) + (2 * n**3 + 4 * n * n * m + 2 * n * m * m + m**3 / 3
                                                                 + 2 * m * m * n)


def dare_grad_flops(n, m, stein_steps):
    """per instance: each Smith step three n x n products (6n^3, the last step skips M^2); around it PA, PB, the gain,
    Yk, Gbar, S (4n^3 + 2n^2 m + ...), Acl, P Acl, P Acl Y (2n^3) and the four gradients"""
    fixed = (2 * n**3 + 2 * n * n * m + 2 * n * m * m + m**3 / 3 + 4 * m * m * n) + 2 * m * m * n + 2 * m * m * n \
        + 2 * n * m * m + 2 * n * n * m + 4 * n**3 + 2 * n * n * m + 2 * n * n * m + 2 * n**3 + 2 * m * n * n \
        + 4 * m * m * n + 2 * n * n * m + 2 * n * n * m + 2 * n * n * m + 2 * n * m * m
    return stein_steps * 6 * n**3 - 2 * n**3 + fixed


def timed(fn):
    """best per-call time (ms) over three windows of at least WINDOW_S each, after a warm-up window"""
    fn()
    torch.cuda.synchronize()
    t0, reps = time.perf_counter(), 0
    while time.perf_counter() - t0 < WINDOW_S:
        fn()
        torch.cuda.synchronize()
        reps += 1
    best = math.inf
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    return best, reps


RHO_MAX = 0.95


def draws(h, n, m, batch):
    """the first `batch` draws of the seed with rho(A - BK) <= RHO_MAX"""
    prob = problems.dare_lti_riccati(n, m, 2, int(batch * 1.5), seed=n + m)
    _, K, _, info = ops.dare_problem(prob, handle=h)
    rho = np.abs(np.linalg.eigvals(prob["A"] - prob["B"] @ K)).max(axis=1)
    keep = np.nonzero((rho <= RHO_MAX) & (info == 0))[0][:batch]
    assert len(keep) == batch, len(keep)
    return {k: prob[k][keep] for k in "ABQR"}


def run_shape(h, n, m, batch, peak_tflops):
    dev = torch.device("cuda")
    prob = draws(h, n, m, batch)
    cmt = lambda x: torch.from_numpy(np.ascontiguousarray(np.swapaxes(x, -1, -2))).to(dev)  # noqa: E731
    A, B, Q, R = (cmt(prob[k]) for k in "ABQR")
    P = torch.empty(batch, n, n, dtype=torch.float64, device=dev)
    K = torch.empty(batch, n, m, dtype=torch.float64, device=dev)
    iters = torch.empty(batch, dtype=torch.int32, device=dev)
    info = torch.empty(batch, dtype=torch.int32, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(5)
    dP = torch.randn(batch, n, n, generator=gen, dtype=torch.float64, device=dev)
    dK = torch.randn(batch, n, m, generator=gen, dtype=torch.float64, device=dev)
    gA, gB, gQ, gR = (torch.empty_like(x) for x in (A, B, Q, R))
    ginfo = torch.empty(batch, dtype=torch.int32, device=dev)

    def fwd():
        ops.dare(h, n, m, batch, A, B, Q, R, P, K, iters, info)

    def grad():
        ops.dare_grad(h, n, m, batch, A, B, R, P, dP, dK, gA, gB, gQ, gR, ginfo)

    t_fwd, reps_fwd = timed(fwd)
    kern_fwd = h.last_kernel
    t_grad, reps_grad = timed(grad)
    kern_grad = h.last_kernel
    assert int(info.ne(0).sum()) == 0 and int(ginfo.ne(0).sum()) == 0
    it = iters.cpu().numpy()
    Kd = K.cpu().numpy().swapaxes(-1, -2)
    # Stein steps of the gradient, from the oracle on 64 instances (the kernel does not report them)
    stein = []
    Pm = P[:64].cpu().numpy().swapaxes(-1, -2)
    dPm, dKm = dP[:64].cpu().numpy().swapaxes(-1, -2), dK[:64].cpu().numpy().swapaxes(-1, -2)
    for i in range(min(64, batch)):
        _, k, _ = od.dare_grad(prob["A"][i], prob["B"][i], prob["R"][i], Pm[i], dPm[i], dKm[i])
        stein.append(k)
    fl_fwd = float(sum(dare_flops(n, m, int(s)) for s in it))
    fl_grad = dare_grad_flops(n, m, float(np.mean(stein))) * batch

    # the alternative: K_0 of an LTI horizon of N knots, N the least with rho^(2(N-1)) <= 1e-12 for the batch's largest
    # rho(A - BK); the K_0 error reached there is recorded (it includes the Riccati kernels' own rounding)
    rho = np.array([np.abs(np.linalg.eigvals(prob["A"][i] - prob["B"][i] @ Kd[i])).max() for i in range(batch)])
    N = max(4, int(math.ceil(math.log(1e-12) / (2 * math.log(rho.max())))) + 1)
    lti = _lib.FLAG_LTI
    x0 = torch.ones(batch, n, dtype=torch.float64, device=dev)
    Z = torch.empty(batch, _lib.num_vars(n, m, N), dtype=torch.float64, device=dev)
    Kr = torch.empty(batch, N - 1, n, m, dtype=torch.float64, device=dev)
    kff = torch.empty(batch, N - 1, m, dtype=torch.float64, device=dev)
    rinfo = torch.empty(batch, dtype=torch.int32, device=dev)
    ops.riccati(h, n, m, N, batch, lti, A, B, Q, R, None, None, Q, None, x0, Z, Kr, kff, rinfo)
    err = ((Kr[:, 0] - K).abs().amax(dim=(1, 2)) / K.abs().amax(dim=(1, 2))).max().item()

    def alt_fwd():
        ops.riccati(h, n, m, N, batch, lti, A, B, Q, R, None, None, Q, None, x0, Z, Kr, kff, rinfo)

    dKN = torch.zeros(batch, N - 1, n, m, dtype=torch.float64, device=dev)
    dKN[:, 0] = dK
    rg = [torch.empty_like(x) for x in (A, B, Q, R)] + [None] * 5  # gA, gB, gQ, gR; no q, r, Qf, qf, x0

    def alt_grad():
        ops.riccati_grad_gains(h, n, m, N, batch, lti, A, B, Q, R, None, None, Q, None, None, None, dKN, None,
                               *rg, rinfo)

    t_alt_fwd, _ = timed(alt_fwd)
    kern_alt_fwd = h.last_kernel
    t_alt_grad, _ = timed(alt_grad)
    assert int(rinfo.ne(0).sum()) == 0
    hist = {int(k): int(v) for k, v in zip(*np.unique(it, return_counts=True))}
    return dict(n=n, m=m, batch=batch, dare_call_ms=round(t_fwd, 4), dare_grad_call_ms=round(t_grad, 4),
                windows_reps=[reps_fwd, reps_grad], dare_kernel=kern_fwd, dare_grad_kernel=kern_grad,
                doubling_steps_histogram=hist, stein_steps_oracle_64=[int(min(stein)), int(max(stein))],
                rho_acl_range=[round(float(rho.min()), 4), round(float(rho.max()), 4)],
                dare_flops=fl_fwd, dare_tflops=round(fl_fwd / (t_fwd * 1e-3) / 1e12, 3),
                dare_frac_of_dfma_peak=round(fl_fwd / (t_fwd * 1e-3) / 1e12 / peak_tflops, 4),
                dare_grad_flops=fl_grad, dare_grad_tflops=round(fl_grad / (t_grad * 1e-3) / 1e12, 3),
                dare_grad_frac_of_dfma_peak=round(fl_grad / (t_grad * 1e-3) / 1e12 / peak_tflops, 4),
                alternative_N=N, alternative_K0_max_rel_err=err, riccati_gains_call_ms=round(t_alt_fwd, 4),
                riccati_kernel=kern_alt_fwd, riccati_grad_gains_call_ms=round(t_alt_grad, 4),
                speedup_forward=round(t_alt_fwd / t_fwd, 2), speedup_gradient=round(t_alt_grad / t_grad, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU only")
    h = _lib.Handle(0)
    h.set_stream(torch.cuda.current_stream().cuda_stream or 1)  # 1 = cudaStreamLegacy, torch's default stream
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    import ctypes as C
    peak = C.c_double(0.0)
    h.call("lqrb_fp64_peak_f64", 0, 0.5, C.byref(peak))
    rows = []
    for n, m, b in SHAPES:
        rows.append(run_shape(h, n, m, b, peak.value))
        torch.cuda.empty_cache()
    out = dict(tool="dare_bench", device=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q,
               fp64_dfma_peak_tflops_measured=round(peak.value, 2), window_s=WINDOW_S, shapes=rows)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
