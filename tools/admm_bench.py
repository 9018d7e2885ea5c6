#!/usr/bin/env python
"""Cost of box-constrained MPC by ADMM (lqrb_admm_cache_f64 / lqrb_admm_solve_f64), device-resident, next to one LTI
lqrb_riccati_f64 call at the same shape, batch and horizon.  Inputs: the stable draws of problems.dare_lti_riccati,
x0 ~ 3 N(0, 1), zero references, and input bounds at a quarter of each instance's largest unconstrained |u| (the
unconstrained solve is an ADMM solve without bounds), so that they bind; rho = 1.  Per shape: the distribution of the
iterations to eps = 1e-6 (cold start), the call time to that eps, the time per iteration from a fixed-count call
(eps = 0, ITERS_FIXED iterations), the cache call, FLOPs and shared-memory bytes counted from the shapes and the
iterations, and the fraction of the FP64 DFMA peak measured in the same run (lqrb_fp64_peak_f64).  Times from CUDA
events: a warm-up window, then the best of three windows of at least 0.35 s.  The card's name and power limit are read
in the same run.  Prints one JSON line (and writes it to --out when given)."""
import argparse
import ctypes as C
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

SHAPES = [(4, 1, 65536), (12, 4, 16384), (32, 8, 4096)]
N = 50
RHO = 1.0
EPS = 1e-6
MAX_ITER = 5000
ITERS_FIXED = 50
WINDOW_S = 0.35


def iter_fmas(n, m, N):
    """FMAs of one iteration: per knot B'p, K'r (2nm), C2 p (n^2), C1 s (m^2) backward; K x, B u (2nm), A x (n^2)
    forward"""
    return (N - 1) * (2 * n * n + 4 * n * m + m * m)


def iter_smem_bytes(n, m, N):
    """shared-memory bytes one iteration reads and writes: one matrix element per FMA, and per knot the vectors of
    admm_kernel (backward: r ref, z, y, q ref, v, g read, d written; forward: d, z, y, umin, umax, v, g, xmin, xmax read,
    u, z, y, x, v, g written)"""
    return 8 * (iter_fmas(n, m, N) + (N - 1) * (12 * m + 10 * n))


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


def run_shape(h, n, m, batch, peak_tflops):
    dev = torch.device("cuda")
    prob = problems.dare_lti_riccati(n, m, N, batch, seed=n + m)
    cmt = lambda x: torch.from_numpy(np.ascontiguousarray(np.swapaxes(x, -1, -2))).to(dev)  # noqa: E731
    A, B, Q, R = (cmt(prob[k]) for k in "ABQR")
    x0 = torch.from_numpy(3.0 * prob["x0"]).to(dev)
    cache = torch.empty(batch, ops.admm_cache_doubles(n, m), dtype=torch.float64, device=dev)
    cinfo = torch.empty(batch, dtype=torch.int32, device=dev)

    def cache_call():
        ops.admm_cache(h, n, m, batch, RHO, A, B, Q, R, cache, cinfo)

    t_cache, _ = timed(cache_call)
    assert int(cinfo.ne(0).sum()) == 0
    Z = torch.empty(batch, _lib.num_vars(n, m, N), dtype=torch.float64, device=dev)
    iters = torch.empty(batch, dtype=torch.int32, device=dev)
    res = torch.empty(batch, 2, dtype=torch.float64, device=dev)
    info = torch.empty(batch, dtype=torch.int32, device=dev)
    ops.admm_solve(h, n, m, N, batch, cache, x0, Z, max_iter=MAX_ITER, eps_pri=EPS, eps_dual=EPS, iters=iters,
                   res=res, info=info)
    U0 = Z[:, :(N - 1) * (n + m)].view(batch, N - 1, n + m)[:, :, n:]
    ub = 0.25 * U0.abs().amax(dim=(1, 2))
    umax = ub[:, None, None].expand(batch, N - 1, m).contiguous()
    umin = -umax

    def solve(max_iter=MAX_ITER, eps=EPS):
        ops.admm_solve(h, n, m, N, batch, cache, x0, Z, umin=umin, umax=umax, max_iter=max_iter, eps_pri=eps,
                       eps_dual=eps, iters=iters, res=res, info=info)

    t_solve, reps = timed(solve)
    kern = h.last_kernel
    it = iters.cpu().numpy()
    inf = info.cpu().numpy()
    U = Z[:, :(N - 1) * (n + m)].view(batch, N - 1, n + m)[:, :, n:]
    active = float(((U.abs() - umax).abs() <= 1e-6 * umax).double().mean())
    t_fixed, _ = timed(lambda: solve(ITERS_FIXED, 0.0))
    t_iter = t_fixed / ITERS_FIXED
    # one LTI Riccati solve at the same shape, batch and horizon
    Zr = torch.empty_like(Z)
    rinfo = torch.empty(batch, dtype=torch.int32, device=dev)

    def riccati():
        ops.riccati(h, n, m, N, batch, _lib.FLAG_LTI, A, B, Q, R, None, None, Q, None, x0, Zr, None, None, rinfo)

    t_ric, _ = timed(riccati)
    kern_ric = h.last_kernel
    fl_iter = 2.0 * iter_fmas(n, m, N) * batch
    per = (2 * n * n + 2 * n * m + m * m + (N - 1) * (6 * n + 6 * m)) * 8
    G = 4 if n <= 4 else 8 if n <= 8 else 16 if n <= 16 else 32
    ipb = min(32 // G, 227 * 1024 // per)
    pct = lambda q: int(np.percentile(it, q))  # noqa: E731
    return dict(n=n, m=m, N=N, batch=batch, rho=RHO, eps=EPS, kernel=kern, smem_bytes_per_instance=per,
                instances_per_block=ipb, blocks_per_sm_by_smem=int(228 * 1024 // (per * ipb + 1024)),
                cache_call_ms=round(t_cache, 4), solve_call_ms=round(t_solve, 4), windows_reps=reps,
                info_counts={int(k): int(v) for k, v in zip(*np.unique(inf, return_counts=True))},
                iters_min_p50_p90_p99_max=[int(it.min()), pct(50), pct(90), pct(99), int(it.max())],
                iters_mean=round(float(it.mean()), 1), active_input_share=round(active, 3),
                fixed_count_iters=ITERS_FIXED, fixed_count_call_ms=round(t_fixed, 4),
                iteration_ms=round(t_iter, 5), riccati_lti_call_ms=round(t_ric, 4), riccati_kernel=kern_ric,
                iteration_over_riccati=round(t_iter / t_ric, 3),
                iteration_flops=fl_iter, iteration_tflops=round(fl_iter / (t_iter * 1e-3) / 1e12, 3),
                iteration_frac_of_dfma_peak=round(fl_iter / (t_iter * 1e-3) / 1e12 / peak_tflops, 4),
                iteration_smem_bytes=iter_smem_bytes(n, m, N) * batch,
                iteration_smem_tbs=round(iter_smem_bytes(n, m, N) * batch / (t_iter * 1e-3) / 1e12, 3))


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
    peak = C.c_double(0.0)
    h.call("lqrb_fp64_peak_f64", 0, 0.5, C.byref(peak))
    rows = []
    for n, m, b in SHAPES:
        rows.append(run_shape(h, n, m, b, peak.value))
        torch.cuda.empty_cache()
    out = dict(tool="admm_bench", device=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q,
               fp64_dfma_peak_tflops_measured=round(peak.value, 2), window_s=WINDOW_S, shapes=rows)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
