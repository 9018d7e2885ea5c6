#!/usr/bin/env python
"""Cost of the constrained-KKT gradient (lqrb_kkt_grad_f64) next to the forward solve (lqrb_kkt_solve_f64),
device-resident, inputs generated on the device with lqr_b200/synthetic.py.  Per shape: forward and gradient-call
times from CUDA events, the gradient kernel's own time from torch.profiler in a separate pass, that kernel's
algorithmic bytes and their fraction of the 6,548 GB/s copy peak of DESIGN §5, and the parity of 16 instances against
the CPU gradient oracle.  Prints one JSON line (and writes it to --out when given)."""
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
# (label, n, m, N, batch): the BASELINE KKT configs 3 (Dubins), 5a-K and 5b-K.  Config 3 runs at its own batch; 5a-K
# and 5b-K at the batches that fit in HBM with the instance-major inputs (3.0 / 7.7 MB per instance), their gradients
# and the solve's scratch at once (16,384 and 4,096 instances would need more than the card's 180 GB)
SHAPES = [("c3_dubins", 3, 2, 201, 262144), ("5aK", 12, 4, 1001, 4096), ("5bK", 64, 16, 101, 2048)]


def grad_kernel_bytes(n, m, N, p, batch):
    """what kkt_grad_kernel must move: every gradient written once (the shapes of Q, R, q, r, A, B, d, C, c) and the
    forward and adjoint solutions read once"""
    K1 = N - 1
    ws = [n + (m if k < N - 1 else 0) for k in range(N)]
    NN, P = N * n + K1 * m, int(p.sum()) + K1 * n
    writes = n * n * N + m * m * K1 + n * N + m * K1 + n * n * K1 + n * m * K1 + n * K1 + \
        sum(int(pk) * w for pk, w in zip(p, ws)) + int(p.sum())
    return 8 * batch * (writes + 2 * (NN + P))


def run_shape(h, label, n, m, N, batch, steps, warmup):
    f = synthetic.dubins_kkt_chunk(batch, 1, 0, N=N) if label.startswith("c3") else \
        synthetic.random_kkt_chunk(n, m, N, batch, 3, 0)
    p = f["p"]
    NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
    dev = torch.device("cuda")
    dz = torch.empty(batch, NN, dtype=torch.float64, device=dev)
    mult = torch.empty(batch, P, dtype=torch.float64, device=dev)
    info = torch.empty(batch, dtype=torch.int32, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    dzb = torch.randn(batch, NN, generator=g, dtype=torch.float64, device=dev)
    mb = torch.randn(batch, P, generator=g, dtype=torch.float64, device=dev)
    grads = [torch.empty_like(f[k]) for k in ("Q", "R")] + [None] + \
        [torch.empty_like(f[k]) for k in ("q", "r", "A", "B", "d")] + [None] + [torch.empty_like(f[k]) for k in ("C", "c")]
    ginfo = torch.empty(batch, dtype=torch.int32, device=dev)
    torch.cuda.empty_cache()  # the generator's temporaries: the library allocates its scratch with cudaMalloc
    free_gb = torch.cuda.mem_get_info()[0] / 1e9

    def fwd():
        ops.kkt_solve(h, n, m, N, batch, p, f["hess_mode"], 0, f["Q"], f["R"], None, f["q"], f["r"], f["A"], f["B"],
                      f["d"], None, f["C"], f["c"], dz, mult, None, info)

    def grad():
        ops.kkt_grad(h, n, m, N, batch, p, f["hess_mode"], 0, f["Q"], f["R"], None, f["A"], f["B"], None, f["C"], dz,
                     mult, dzb, mb, *grads, ginfo)

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
    t_fwd = timed(fwd)
    fwd_kernel = h.last_kernel
    t_grad = timed(grad)
    kernel_name = h.last_kernel
    assert int(info.ne(0).sum()) == 0 and int(ginfo.ne(0).sum()) == 0

    # the gradient kernel's own time, profiler on, in a pass of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            grad()
        torch.cuda.synchronize()
    ks = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    t_kern = sum(e.device_time for e in ks if "kkt_grad_kernel" in e.name) / steps / 1e3  # ms
    t_kernels = {}
    for e in ks:
        key = e.name.split("<")[0].split("(")[0]
        t_kernels[key] = t_kernels.get(key, 0.0) + e.device_time / steps / 1e3
    nbytes = grad_kernel_bytes(n, m, N, p, batch)

    # parity of 16 instances against the oracle
    from oracle.kkt_grad import kkt_grad
    cnt = 16
    go = kkt_grad(synthetic.kkt_to_math(f, 0, cnt), dzb[:cnt].cpu().numpy(), mb[:cnt].cpu().numpy())
    got, _ = ops.kkt_grad_problem(synthetic.kkt_to_math(f, 0, cnt), dz[:cnt].cpu().numpy(), mult[:cnt].cpu().numpy(),
                                  dzb[:cnt].cpu().numpy(), mb[:cnt].cpu().numpy(), handle=h)
    worst = 0.0
    for k in ("Q", "R", "q", "r", "A", "B", "d"):
        worst = max(worst, float(np.linalg.norm(got[k] - go[k]) / np.linalg.norm(go[k])))
    for k in ("C", "c"):
        a, b = (np.concatenate([x.reshape(cnt, -1) for x in v], axis=1) for v in (got[k], go[k]))
        worst = max(worst, float(np.linalg.norm(a - b) / np.linalg.norm(b)))
    return dict(shape=label, n=n, m=m, N=N, batch=batch, forward_ms=round(t_fwd, 4), grad_call_ms=round(t_grad, 4),
                grad_over_forward=round(t_grad / t_fwd, 3), grad_kernel_ms=round(t_kern, 4), grad_kernel_bytes=nbytes,
                grad_kernel_gbs=round(nbytes / (t_kern * 1e-3) / 1e9, 1),
                grad_kernel_frac_copy_peak=round(nbytes / (t_kern * 1e-3) / 1e9 / COPY_PEAK_GBS, 3),
                kernels_ms={k: round(v, 4) for k, v in sorted(t_kernels.items())},
                forward_kernel=fwd_kernel, kernel=kernel_name, parity_16_max_rel_err=worst,
                device_free_gb_before_calls=round(free_gb, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU only")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    rows = []
    for s in SHAPES:
        if s[0] in a.shapes.split(","):
            h = _lib.Handle(0)  # a handle per shape: its grow-only scratch is freed before the next shape
            h.set_stream(torch.cuda.current_stream().cuda_stream or 1)  # 1 = cudaStreamLegacy, torch's default stream
            rows.append(run_shape(h, *s, a.steps, a.warmup))
            h.close()
            torch.cuda.empty_cache()
    out = dict(tool="kkt_grad_bench", device=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q,
               copy_peak_gbs=COPY_PEAK_GBS, steps=a.steps, warmup=a.warmup, shapes=rows)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
