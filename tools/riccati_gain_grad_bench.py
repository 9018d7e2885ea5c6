#!/usr/bin/env python
"""Cost of the gradient through the Riccati gains (lqrb_riccati_grad_gains_f64) next to the forward solve with K and
kff (lqrb_riccati_f64), device-resident, inputs generated on the device with lqr_b200/synthetic.py.  Per shape: the
forward call, the new call with gain cotangents only and with dZ, dK, dkff, from CUDA events; the gain kernel's own
time from torch.profiler in a separate pass; its FLOPs and bytes from the shapes, and their fraction of the FP64 DFMA
peak (33.8 TFLOP/s, profiles/r1_fp64_peak_ubench.json) or of the 6,548 GB/s copy peak, whichever bounds it; and the
parity of 64 instances against the CPU oracle.  Prints one JSON line (and writes it to --out when given)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lqr_b200 import _lib, ops, synthetic  # noqa: E402

COPY_PEAK_GBS = 6548.2
FP64_PEAK_TFLOPS = 33.8
NAMES = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")
# the shapes of tools/riccati_grad_bench.py: config 2 (cartpole) LTV-affine and LTI; 5a-R at a long horizon; 5b-R
SHAPES = [("cartpole_ltv", 4, 1, 101, 65536, False), ("cartpole_lti", 4, 1, 101, 65536, True),
          ("12x4_N1001", 12, 4, 1001, 4096, False), ("64x16_N101", 64, 16, 101, 2048, False)]


def gain_kernel_flops(n, m, N, batch):
    """multiply-adds x 2 of riccati_gain_grad_kernel per knot (DESIGN §4.10), m^3 / 3 for the factor of G"""
    solve = 2 * (n + 1) * m * m  # n + 1 rows through L and L'
    back = 2 * (2 * n**3 + 3 * n * n * m + n * m * m + n * n + n * m) + m**3 / 3 + solve
    fwd = 2 * (3 * n**3 + 9 * n * n * m + 4 * n * m * m + 6 * n * n + 4 * n * m) + solve
    return (N - 1) * batch * (back + fwd)


def gain_kernel_bytes(n, m, N, batch, lti):
    """what the kernel must move: A, B, Q, R, q, r (per knot, or once under LTI), Qf, qf, dK, dkff read; the tape written
    and read back; every gradient read and written (it adds into the Z part)"""
    Kn = 1 if lti else N - 1
    tape = (N - 1) * (n * n + n + m * n + m + m * m)
    inputs = Kn * (2 * n * n + n * m + m * m + n + m) + n * n + n + (N - 1) * (m * n + m)
    grads = Kn * (2 * n * n + n * m + m * m + n + m) + n * n + n
    return 8 * batch * (inputs + 2 * tape + 2 * grads)


def make(n, m, N, batch, lti, seed=0):
    f = synthetic.riccati_cartpole_chunk(batch, seed, 0, N=N) if n == 4 else \
        synthetic.random_riccati_chunk(n, m, N, batch, seed, 0)
    if lti:  # knot 0 of every per-knot array
        for k in ("A", "B", "Q", "R", "q", "r"):
            f[k] = f[k][:, 0].contiguous()
    return f


def run_shape(h, label, n, m, N, batch, lti, steps, warmup):
    f = make(n, m, N, batch, lti)
    flags = _lib.FLAG_LTI if lti else 0
    NN = _lib.num_vars(n, m, N)
    dev = torch.device("cuda")
    Z = torch.empty(batch, NN, dtype=torch.float64, device=dev)
    K = torch.empty(batch, N - 1, n, m, dtype=torch.float64, device=dev)
    kff = torch.empty(batch, N - 1, m, dtype=torch.float64, device=dev)
    info = torch.empty(batch, dtype=torch.int32, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    dZ = torch.randn(batch, NN, generator=g, dtype=torch.float64, device=dev)
    dK = torch.randn(batch, N - 1, n, m, generator=g, dtype=torch.float64, device=dev)
    dkff = torch.randn(batch, N - 1, m, generator=g, dtype=torch.float64, device=dev)
    grads = [torch.empty_like(f[k]) for k in NAMES]
    ginfo = torch.empty(batch, dtype=torch.int32, device=dev)
    ins = [f[k] for k in ("A", "B", "Q", "R", "q", "r", "Qf", "qf")]

    def fwd():
        ops.riccati(h, n, m, N, batch, flags, *ins, f["x0"], Z, K, kff, info)

    def gains_only():
        ops.riccati_grad_gains(h, n, m, N, batch, flags, *ins, None, None, dK, dkff, *grads, ginfo)

    def all_three():
        ops.riccati_grad_gains(h, n, m, N, batch, flags, *ins, Z, dZ, dK, dkff, *grads, ginfo)

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    t_fwd, t_gains, t_all = timed(fwd), timed(gains_only), timed(all_three)
    kernel_name = h.last_kernel
    assert int(info.ne(0).sum()) == 0 and int(ginfo.ne(0).sum()) == 0

    # the gain kernel's own time, profiler on, in a pass of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            gains_only()
        torch.cuda.synchronize()
    ks = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    t_kern = sum(e.device_time for e in ks if "riccati_gain_grad_kernel" in e.name) / steps / 1e3  # ms
    flops, nbytes = gain_kernel_flops(n, m, N, batch), gain_kernel_bytes(n, m, N, batch, lti)
    t_flop, t_byte = flops / (FP64_PEAK_TFLOPS * 1e12), nbytes / (COPY_PEAK_GBS * 1e9)
    bound = "fp64" if t_flop >= t_byte else "copy"

    # parity of 64 instances (all three cotangents) against the oracle
    from oracle.riccati_gain_grad import riccati_total_grad
    all_three()
    torch.cuda.synchronize()
    cnt = 64
    if lti:
        sw = lambda a: np.ascontiguousarray(np.swapaxes(a[:cnt].cpu().numpy(), -1, -2))  # noqa: E731
        prob = dict(n=n, m=m, N=N, lti=True, A=sw(f["A"]), B=sw(f["B"]), Q=sw(f["Q"]), R=sw(f["R"]),
                    q=f["q"][:cnt].cpu().numpy(), r=f["r"][:cnt].cpu().numpy(), Qf=sw(f["Qf"]),
                    qf=f["qf"][:cnt].cpu().numpy(), x0=f["x0"][:cnt].cpu().numpy())
    else:
        prob = synthetic.riccati_to_math(f, 0, cnt)
    go = riccati_total_grad(prob, dZ[:cnt].cpu().numpy(), np.swapaxes(dK[:cnt].cpu().numpy(), -1, -2),
                            dkff[:cnt].cpu().numpy())
    worst = 0.0
    for k, t in zip(NAMES, grads):
        a = t[:cnt].cpu().numpy()
        if k in ("A", "B", "Q", "R", "Qf"):
            a = np.swapaxes(a, -1, -2)
        worst = max(worst, float(np.linalg.norm(a - go[k]) / np.linalg.norm(go[k])))
    return dict(shape=label, n=n, m=m, N=N, batch=batch, lti=lti, forward_with_gains_ms=round(t_fwd, 4),
                gains_only_call_ms=round(t_gains, 4), all_three_call_ms=round(t_all, 4),
                gains_only_over_forward=round(t_gains / t_fwd, 3), all_three_over_forward=round(t_all / t_fwd, 3),
                gain_kernel_ms=round(t_kern, 4), gain_kernel_flops=flops, gain_kernel_bytes=nbytes,
                gain_kernel_tflops=round(flops / (t_kern * 1e-3) / 1e12, 3),
                gain_kernel_gbs=round(nbytes / (t_kern * 1e-3) / 1e9, 1), bound=bound,
                gain_kernel_frac_of_bound_peak=round(max(t_flop, t_byte) / (t_kern * 1e-3), 3),
                kernel=kernel_name, parity_64_max_rel_err=worst)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU only")
    h = _lib.Handle(0)
    h.set_stream(torch.cuda.current_stream().cuda_stream or 1)  # 1 = cudaStreamLegacy, torch's default stream
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    rows = []
    for s in SHAPES:
        if s[0] in a.shapes.split(","):
            rows.append(run_shape(h, *s, a.steps, a.warmup))
            torch.cuda.empty_cache()
    out = dict(tool="riccati_gain_grad_bench", device=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q,
               copy_peak_gbs=COPY_PEAK_GBS, fp64_peak_tflops=FP64_PEAK_TFLOPS, steps=a.steps, warmup=a.warmup,
               shapes=rows)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
