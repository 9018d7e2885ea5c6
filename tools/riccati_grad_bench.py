#!/usr/bin/env python
"""Cost of the Riccati gradient (lqrb_riccati_grad_f64) next to the forward solve (lqrb_riccati_f64), device-resident,
inputs generated on the device with lqr_b200/synthetic.py.  Per shape: forward and gradient-call times from CUDA
events, the gradient kernel's own time from torch.profiler in a separate pass, that kernel's algorithmic bytes and
their fraction of the 6,548 GB/s copy peak of DESIGN §5, and the parity of 64 instances against the CPU gradient
oracle.  Prints one JSON line (and writes it to --out when given)."""
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
NAMES = ("A", "B", "Q", "R", "q", "r", "Qf", "qf", "x0")
# (label, n, m, N, batch, lti): config 2 (cartpole) LTV-affine and LTI; 5a-R at a long horizon; 5b-R
SHAPES = [("cartpole_ltv", 4, 1, 101, 65536, False), ("cartpole_lti", 4, 1, 101, 65536, True),
          ("12x4_N1001", 12, 4, 1001, 4096, False), ("64x16_N101", 64, 16, 101, 2048, False)]


def grad_kernel_bytes(n, m, N, batch, lti):
    """what the sweep must move: reads A, B, Q, R, q, r per knot (Kn of them), K_k for every knot, Qf, qf, Z, Z^, dZ;
    writes every gradient"""
    Kn = 1 if lti else N - 1
    NN = N * n + (N - 1) * m
    reads = Kn * (2 * n * n + n * m + m * m + n + m) + (N - 1) * m * n + n * n + n + 3 * NN
    writes = Kn * (2 * n * n + n * m + m * m + n + m) + n * n + 2 * n
    return 8 * batch * (reads + writes)


def make(label, n, m, N, batch, lti, seed=0):
    f = synthetic.riccati_cartpole_chunk(batch, seed, 0, N=N) if n == 4 else \
        synthetic.random_riccati_chunk(n, m, N, batch, seed, 0)
    if lti:  # knot 0 of every per-knot array
        for k in ("A", "B", "Q", "R", "q", "r"):
            f[k] = f[k][:, 0].contiguous()
    return f


def run_shape(h, label, n, m, N, batch, lti, steps, warmup):
    f = make(label, n, m, N, batch, lti)
    flags = _lib.FLAG_LTI if lti else 0
    NN = _lib.num_vars(n, m, N)
    dev = torch.device("cuda")
    Z = torch.empty(batch, NN, dtype=torch.float64, device=dev)
    info = torch.empty(batch, dtype=torch.int32, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    dZ = torch.randn(batch, NN, generator=g, dtype=torch.float64, device=dev)
    grads = [torch.empty_like(f[k]) for k in NAMES]
    ginfo = torch.empty(batch, dtype=torch.int32, device=dev)
    ins = [f[k] for k in ("A", "B", "Q", "R", "q", "r", "Qf", "qf")]

    def fwd():
        ops.riccati(h, n, m, N, batch, flags, *ins, f["x0"], Z, None, None, info)

    def grad():
        ops.riccati_grad(h, n, m, N, batch, flags, *ins, Z, dZ, *grads, ginfo)

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
    t_fwd, t_grad = timed(fwd), timed(grad)
    kernel_name = h.last_kernel
    assert int(info.ne(0).sum()) == 0 and int(ginfo.ne(0).sum()) == 0

    # the gradient kernel's own time, profiler on, in a pass of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            grad()
        torch.cuda.synchronize()
    ks = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    t_kern = sum(e.device_time for e in ks if "riccati_grad_kernel" in e.name) / steps / 1e3  # ms
    t_kernels = {}
    for e in ks:
        key = e.name.split("<")[0].split("(")[0]
        t_kernels[key] = t_kernels.get(key, 0.0) + e.device_time / steps / 1e3
    nbytes = grad_kernel_bytes(n, m, N, batch, lti)

    # parity of 64 instances against the oracle
    from oracle.riccati_grad import riccati_grad
    cnt = 64
    prob = synthetic.riccati_to_math(f, 0, cnt) if not lti else None
    if lti:
        sw = lambda a: np.ascontiguousarray(np.swapaxes(a[:cnt].cpu().numpy(), -1, -2))  # noqa: E731
        prob = dict(n=n, m=m, N=N, lti=True, A=sw(f["A"]), B=sw(f["B"]), Q=sw(f["Q"]), R=sw(f["R"]),
                    q=f["q"][:cnt].cpu().numpy(), r=f["r"][:cnt].cpu().numpy(), Qf=sw(f["Qf"]),
                    qf=f["qf"][:cnt].cpu().numpy(), x0=f["x0"][:cnt].cpu().numpy())
    go = riccati_grad(prob, dZ[:cnt].cpu().numpy())
    worst = 0.0
    for k, t in zip(NAMES, grads):
        a = t[:cnt].cpu().numpy()
        if k in ("A", "B", "Q", "R", "Qf"):
            a = np.swapaxes(a, -1, -2)
        worst = max(worst, float(np.linalg.norm(a - go[k]) / np.linalg.norm(go[k])))
    return dict(shape=label, n=n, m=m, N=N, batch=batch, lti=lti, forward_ms=round(t_fwd, 4),
                grad_call_ms=round(t_grad, 4), grad_over_forward=round(t_grad / t_fwd, 3),
                grad_kernel_ms=round(t_kern, 4), grad_kernel_bytes=nbytes,
                grad_kernel_gbs=round(nbytes / (t_kern * 1e-3) / 1e9, 1),
                grad_kernel_frac_copy_peak=round(nbytes / (t_kern * 1e-3) / 1e9 / COPY_PEAK_GBS, 3),
                kernels_ms={k: round(v, 4) for k, v in sorted(t_kernels.items())},
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
    out = dict(tool="riccati_grad_bench", device=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q,
               copy_peak_gbs=COPY_PEAK_GBS, steps=a.steps, warmup=a.warmup, shapes=rows)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
