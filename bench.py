#!/usr/bin/env python
"""bench.py — batched LQR KKT solves/sec (FP64) on B200, the BASELINE.json metric, for EVERY BASELINE config.

Headline (`value`, `e2e`, `roofline`, `cpu_baseline` at the top level of the JSON line): BASELINE.json configs[1] —
batched cartpole LQR n=4 m=1 N=101, 65,536 random LTV-affine instances per GPU, Riccati backward pass + forward
rollout (SURVEY §8d config 2).  A "step" = one pass of the hot path over the whole batch; weak scaling (per-GPU
work fixed as N grows, batch slices, no collective on the data path).

  value : solves/s with the packed inputs already resident in HBM (one kernel launch per step), CUDA-event timed
          on the launching stream, max over ranks.
  e2e   : the same metric through the reference-facing C-ABI call lqrb_riccati_f64 with HOST (pinned)
          instance-major buffers: H2D + pack + solve + unpack + D2H inside the timed region.
  configs : one entry per BASELINE config (1, 2, 3, 4, 5a-R, 5a-K, 5b-R, 5b-K), each with its own value,
          ms_per_step, clocks sampled while it ran, roofline {bound, achieved, peak, frac, traffic}, kernel name and
          `parity` = worst relative error of >= 64 instances of the TIMED output against the CPU oracle (and
          against the extended-precision global KKT solve for instance 0).  Same harness as the reference's
          LQR.benchmark_solve! (src/LQR.jl:29-36, used at test/cholesky_comp.jl:23-24): identical problem, solve
          repeated, solution checked.  All instances are distinct (seeded device generators, lqr_b200.synthetic).
  fp64_peak : DFMA / DMMA throughput measured in this run (lqrb_fp64_peak_f64) — the denominator of the FP64-bound
          fractions, with its own clock record.

  --steps K / --warmup W : every config runs W untimed steps (at least 3), then exactly K timed steps.
  --dump-outputs DIR : after the timed steps, each config's outputs of its last step as DIR/<config key>_<name>.npy
          (float64; a fixed seeded sample of instances, 60 MiB in all).  The inputs depend only on the arguments, so
          two builds of the library can be compared output for output.

  --impl reference : times the reference algorithm's CPU restatement (oracle/, OpenMP over all host cores) on a
          bounded sample of the same workloads.  (LQR.jl itself is pure Julia and Julia is not installed in this
          image — see DESIGN.md.)
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "batched LQR KKT solves/sec (FP64)"
UNIT = "solves/s"
PARITY_INSTANCES = 64
DUMP_BYTES = 60 << 20   # --dump-outputs: total size of the written sample, shared equally by the configs that run

# key, BASELINE config, workload name, kind, n, m, N, per-GPU batch, roofline bound, parity tolerance
CONFIGS = [
    dict(key="c2", baseline_config=2, workload="cartpole_riccati_n4_m1_N101_b65536", kind="riccati", gen="cartpole",
         n=4, m=1, N=101, batch=65536, bound="hbm", tol=1e-10, seed=0),
    dict(key="c1", baseline_config=1, workload="cartpole_fixture_kkt_n4_m1_N101_b1", kind="fixture",
         n=4, m=1, N=101, batch=1, bound="latency", tol=1e-10, seed=0),
    dict(key="c3", baseline_config=3, workload="dubins_kkt_n3_m2_N201_b262144", kind="kkt", gen="dubins",
         n=3, m=2, N=201, batch=262144, bound="hbm", tol=1e-10, seed=1),
    dict(key="c4", baseline_config=4, workload="dubins_sqp_x10_n3_m2_N201_b65536", kind="sqp",
         n=3, m=2, N=201, batch=65536, bound="hbm", tol=1e-6, seed=2),
    dict(key="5aR", baseline_config=5, workload="quad_riccati_n12_m4_N1001_b16384", kind="riccati", gen="random",
         n=12, m=4, N=1001, batch=16384, bound="hbm", tol=1e-10, seed=3),
    dict(key="5aK", baseline_config=5, workload="quad_kkt_n12_m4_N1001_b16384", kind="kkt", gen="random",
         n=12, m=4, N=1001, batch=16384, bound="fp64", tol=1e-10, seed=3),
    dict(key="5bR", baseline_config=5, workload="large_riccati_n64_m16_N101_b4096", kind="riccati", gen="random",
         n=64, m=16, N=101, batch=4096, bound="fp64", tol=1e-10, seed=4),
    dict(key="5bK", baseline_config=5, workload="large_kkt_n64_m16_N101_b4096", kind="kkt", gen="random",
         n=64, m=16, N=101, batch=4096, bound="fp64", tol=1e-10, seed=4),
]
HEADLINE = "c2"


def tri(k):
    return k * (k + 1) // 2


def riccati_bytes(n, m, N):
    """SURVEY §8d: unique FP64 words read once + written once per instance (symmetric packed)."""
    words_in = (N - 1) * (n * n + n * m + tri(n) + tri(m) + n + m) + tri(n) + 2 * n
    return 8 * (words_in + N * n + (N - 1) * m)


def riccati_flops(n, m, N):
    return (N - 1) * (4 * n**3 + 8 * n * n * m + 4 * n * m * m + m**3 / 3 + 2 * n * n + 4 * n * m)


def kkt_flops(n, m, N, p):
    """SURVEY §8d, the reference's op sequence: shur! (a12) + block-tridiagonal cholesky! (a14) + the two
    substitutions (a15-16) + calc_primals! (a17), per knot."""
    t = 0.0
    for k in range(N):
        w = n + (m if k < N - 1 else 0)
        p1, ps, p2 = (n if k > 0 else 0), int(p[k]), (n if k < N - 1 else 0)
        rho = p1 + ps + p2
        t += w**3 / 3 + 2 * w * w * rho + 2 * rho * rho * w + 2 * rho * w
        t += (p1 * p1 * ps + 2 * p1 * ps * ps + ps**3 / 3 + p1 * p1 * p2 + 2 * ps * p1 * p2 + ps * ps * p2
              + 2 * p1 * p2 * p2 + 2 * ps * p2 * p2 + p2**3 / 3)
        t += 4 * (ps * ps + p2 * p2 + p1 * ps + p1 * p2 + ps * p2)
        t += 2 * rho * w + 2 * w * w
    return t


# ------------------------------------------------------------------ clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return self
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()
        return self

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append((time.perf_counter(), parts))

    def mark(self):
        return time.perf_counter()

    def stop(self, t0=None, t1=None):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        return self.window(t0, t1)

    def window(self, t0=None, t1=None):
        """Median SM clock and throttle reasons of the samples taken in [t0, t1] (all samples if None)."""
        sm, smax, reasons = [], [], set()
        for ts, p in list(self.samples):
            if t0 is not None and (ts < t0 or ts > t1):
                continue
            try:
                sm.append(float(p[0]))
                smax.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ peaks / committed ncu traffic
def measured_peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured copy bandwidth (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload, kernel_name):
    """dram bytes read+written per step of the timed kernels, from the committed `ncu --set full` capture of this
    workload — reported only while the capture is of the SAME kernel that ran (a changed kernel makes it stale)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            e = json.load(f).get(workload)
    except Exception:
        return None, None
    if not isinstance(e, dict) or e.get("kernel") != kernel_name:
        return None, None
    return e.get("bytes"), e.get("source")


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ------------------------------------------------------------------ CPU legs (oracle port) — reference arm and cpu_baseline
def cpu_problem(cfg, count):
    """Seeded host instances of a config for the CPU legs (numpy generators of lqr_b200.problems)."""
    from lqr_b200 import problems
    n, m, N = cfg["n"], cfg["m"], cfg["N"]
    if cfg["kind"] == "riccati":
        return (problems.riccati_cartpole_batch(count, seed=cfg["seed"], N=N) if cfg["gen"] == "cartpole"
                else problems.random_lqr_riccati(n, m, N, count, seed=cfg["seed"]))
    if cfg["kind"] == "kkt":
        return (problems.dubins_kkt_batch(count, seed=cfg["seed"], N=N) if cfg["gen"] == "dubins"
                else problems.random_lqr_kkt(n, m, N, count, seed=cfg["seed"], mid_p=0))
    if cfg["kind"] == "fixture":
        return problems.cartpole_fixture(N)
    raise ValueError(cfg["kind"])


def cpu_time_config(cfg, target_seconds, steps=1, warmup=0):
    """Times the oracle's OpenMP batch driver (the reference algorithm's C restatement) on a bounded sample of a
    config.  Returns dict(value, cores, sample, ms_per_step)."""
    import oracle
    oracle.build()
    cores = host_cores()
    kind = cfg["kind"]
    if kind == "sqp":
        from oracle import sqp_dubins as S
        cnt = 32
        Z0, x0, xf, o = S.turn90_problem(cnt, N=cfg["N"], seed=cfg["seed"])
        t0 = time.perf_counter()
        _, _, _, _, solves = S.solve(Z0, x0, xf, o)
        t = time.perf_counter() - t0
        return dict(value=solves / t, cores=cores, ms_per_step=1e3 * t,
                    sample=f"{cnt} instances x 10 SQP iterations = {solves} KKT solves, 1 step (numpy loop around "
                           f"the OpenMP KKT chain)")
    probe = {"c2": 2048, "c1": 1, "c3": 1024, "5aR": 32, "5aK": 32, "5bR": 16, "5bK": 16}[cfg["key"]]
    cap = {"c2": 16384, "c1": 1, "c3": 4096, "5aR": 128, "5aK": 128, "5bR": 64, "5bK": 64}[cfg["key"]]
    prob = cpu_problem(cfg, cap)
    if kind == "riccati":
        from lqr_b200 import ops
        f = ops.riccati_flatten(prob)
        n, m, N = cfg["n"], cfg["m"], cfg["N"]

        def run(cnt):
            X = np.zeros((cnt, N, n)); U = np.zeros((cnt, N - 1, m))
            K = np.zeros((cnt, N - 1, n, m)); kff = np.zeros((cnt, N - 1, m))
            info = np.zeros(cnt, dtype=np.int32)
            t0 = time.perf_counter()
            oracle.riccati_raw(n, m, N, 0, cnt, f["A"][:cnt], f["B"][:cnt], f["Q"][:cnt], f["R"][:cnt], f["q"][:cnt],
                               f["r"][:cnt], f["Qf"][:cnt], f["qf"][:cnt], f["x0"][:cnt], X, U, K, kff, info, cores)
            return time.perf_counter() - t0
    else:
        f = oracle.kkt_flatten(prob)

        def run(cnt):
            g = dict(f)
            g["batch"] = cnt
            for k in ("Q", "R", "Hux", "q", "r", "A", "B", "d", "D2", "C", "c"):
                if g[k] is not None:
                    g[k] = g[k][:cnt]
            t0 = time.perf_counter()
            oracle.kkt_solve(g, nthreads=cores)
            return time.perf_counter() - t0
    probe = min(probe, cap)
    run(probe)
    t_probe = run(probe)
    per_step = max(1, steps + warmup)
    cnt = int(min(cap, max(probe, probe * (target_seconds / per_step) / max(t_probe, 1e-6))))
    for _ in range(warmup):
        run(cnt)
    times = [run(cnt) for _ in range(max(1, steps))]
    t = sum(times) / len(times)
    return dict(value=cnt / t, cores=cores, ms_per_step=1e3 * t,
                sample=f"{cnt} of {cfg['batch']} instances per step, {len(times)} step(s)")


def sparse_leg(n, m, N, seed, seconds=3.0, max_inst=256):
    """The reference's other solver on the same instances: SparseSolver assembles the global KKT pieces and calls
    a sparse factorisation (src/sparse_solver.jl:267-292).  Analogue here: scipy's sparse LU of [H D'; D 0] per
    instance (assembly excluded), one core, bounded sample.  Reported next to the block-recursion port."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    from lqr_b200 import problems
    from oracle import dense_kkt
    prob = dense_kkt.riccati_as_kkt(problems.riccati_cartpole_batch(max_inst, seed=seed, N=N))
    t_solve, cnt = 0.0, 0
    while cnt < max_inst and t_solve < seconds:
        H, g, D, d = dense_kkt.assemble(prob, cnt)
        K = sp.bmat([[H, D.T], [D, None]], format="csc")
        rhs = -np.concatenate([g, d])
        t0 = time.perf_counter()
        spla.splu(K).solve(rhs)
        t_solve += time.perf_counter() - t0
        cnt += 1
    return {"value": cnt / t_solve, "unit": UNIT, "cores": 1, "sample": f"{cnt} instances",
            "what": "scipy sparse LU of the assembled KKT system (analogue of src/sparse_solver.jl:267-292)"}


# ------------------------------------------------------------------ parity of the timed output (oracle = checker)
def _rel_rows(a, b):
    """worst per-instance relative 2-norm error."""
    num = np.linalg.norm(a - b, axis=1)
    den = np.maximum(np.linalg.norm(b, axis=1), 1e-300)
    return float((num / den).max())


def parity_riccati(prob_math, Z, n, m, N):
    import oracle
    from lqr_b200 import ops
    from oracle import dense_kkt
    oracle.build()
    Xo, Uo, _, _, io = oracle.riccati(prob_math)
    X, U = ops.split_primals(Z, n, m, N)
    b = Z.shape[0]
    e = max(_rel_rows(X.reshape(b, -1), Xo.reshape(b, -1)), _rel_rows(U.reshape(b, -1), Uo.reshape(b, -1)))
    zt, _ = dense_kkt.kkt_truth(dense_kkt.riccati_as_kkt(prob_math), 0)   # extended-precision global KKT solve
    et = float(np.linalg.norm(Z[0] - zt) / np.linalg.norm(zt))
    return dict(max_rel_err=e, vs="oracle/lqr_oracle.c riccati", instances=b, refined_truth_rel_err=et,
                oracle_info_ok=bool((io == 0).all()))


def parity_kkt(prob_math, dz, mult):
    import oracle
    from oracle import dense_kkt
    oracle.build()
    dzo, lamo, io = oracle.kkt_solve(prob_math)
    e = max(_rel_rows(dz, dzo), _rel_rows(mult, lamo))
    zt, lt = dense_kkt.kkt_truth(prob_math, 0)
    et = max(float(np.linalg.norm(dz[0] - zt) / np.linalg.norm(zt)), float(np.linalg.norm(mult[0] - lt) / np.linalg.norm(lt)))
    rs, rp = dense_kkt.kkt_residuals(prob_math, 0, dz[0], mult[0])
    return dict(max_rel_err=e, vs="oracle/lqr_oracle.c kkt chain", instances=dz.shape[0], refined_truth_rel_err=et,
                kkt_residuals_instance0=[rs, rp], oracle_info_ok=bool((io == 0).all()))


# ------------------------------------------------------------------ GPU arm: one config
class Runner:
    def __init__(self, args, rank, local_rank, world):
        import torch
        self.torch = torch
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        self.sampler = ClockSampler(local_rank).start()
        self.hbm_peak, self.hbm_src = measured_peak_hbm()
        self.fp64_peak = None
        self.launches_timed = 0
        self.dump_share = DUMP_BYTES  # main() divides it among the configs that run

    def handle(self):
        from lqr_b200 import _lib
        h = _lib.Handle(self.local_rank)
        # a real (non-default) stream: the handle launches on it and the CUDA events are recorded on it
        h.set_stream(self.stream.cuda_stream)
        return h

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def time_steps(self, h, step, steps, warmup, min_clock_window_s=0.35):
        """W untimed steps, then exactly `steps` steps bracketed by barrier + synchronize, one CUDA event per step on
        the launching stream.  The clock window = warm-up + timed region (+ the same launches repeated afterwards
        until the window is long enough for a few 50-ms nvidia-smi samples; those extra launches are not timed)."""
        torch = self.torch
        t_w0 = self.sampler.mark()
        for _ in range(warmup):
            step()
        self.barrier()
        l0 = h.launches
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record(self.stream)
        for i in range(steps):
            step()
            ev[i + 1].record(self.stream)
        self.barrier()
        launches = h.launches - l0
        total_ms = ev[0].elapsed_time(ev[-1])
        per = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        while self.sampler.mark() - t_w0 < min_clock_window_s:
            step()
            torch.cuda.synchronize()
        t_w1 = self.sampler.mark()
        time.sleep(0.06)
        return total_ms, per, launches, self.sampler.window(t_w0, t_w1)

    def dump_outputs(self, cfg, arrays):
        """--dump-outputs: what the last timed step of a config computed.  `arrays` maps an output's name to a device
        tensor with one row per instance; each is written as DIR/<config key>_<name>.npy in float64.  Outputs larger
        than the config's share of DUMP_BYTES are represented by a fixed seeded sample of instances, the same on every
        run with the same arguments; DIR/<config key>_instances.npy lists the instances written.  (The untimed steps
        time_steps may append for the clock record repeat the last step on the same inputs, bit for bit.)"""
        torch = self.torch
        first = next(iter(arrays.values()))
        batch = first.shape[0]
        per_instance = 8 * (1 + sum(t[0].numel() for t in arrays.values()))
        count = max(1, min(batch, self.dump_share // per_instance))
        idx = (np.arange(batch) if count == batch
               else np.sort(np.random.default_rng(0).choice(batch, size=count, replace=False)))
        sel = torch.from_numpy(idx).to(first.device)
        out = {"instances": idx}
        out.update({name: t.index_select(0, sel).cpu().numpy() for name, t in arrays.items()})
        os.makedirs(self.args.dump_outputs, exist_ok=True)
        for name, a in out.items():
            np.save(os.path.join(self.args.dump_outputs, f"{cfg['key']}_{name}.npy"), a.astype(np.float64))

    def dumping(self):
        return bool(self.args.dump_outputs) and self.rank == 0

    # ---------------------------------------------------------------- fp64 peak
    def measure_fp64_peak(self):
        import ctypes as C
        from lqr_b200 import _lib
        h = self.handle()
        out = {}
        t0 = self.sampler.mark()
        for kind, name in ((0, "dfma_tflops"), (1, "dmma_m8n8k4_tflops")):
            v = C.c_double(0.0)
            h.call("lqrb_fp64_peak_f64", kind, 0.4, C.byref(v))
            out[name] = v.value
        t1 = self.sampler.mark()
        time.sleep(0.06)
        out["clocks"] = self.sampler.window(t0, t1)
        out["how"] = "lqrb_fp64_peak_f64: register-only DFMA / mma.sync.m8n8k4.f64 kernels, best launch of 0.4 s each"
        h.close()
        _ = _lib
        self.fp64_peak = out
        return out

    # ---------------------------------------------------------------- roofline of one config
    def roofline(self, cfg, kernel_ms, batch, bytes_per, flops_per, kernel, workload):
        traffic, src = ncu_traffic(workload, kernel)
        r = {"kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes_per_solve": bytes_per,
             "algorithmic_flops_per_solve": flops_per, "traffic": traffic, "traffic_source": src}
        gbs = bytes_per * batch / (kernel_ms * 1e-3) / 1e9
        tfs = flops_per * batch / (kernel_ms * 1e-3) / 1e12
        if cfg["bound"] == "fp64":
            peak = (self.fp64_peak or {}).get("dmma_m8n8k4_tflops") or 37.2
            r.update(bound="tensor", achieved=tfs, peak=peak, unit="TFLOP/s", frac=tfs / peak,
                     peak_source="FP64 DMMA throughput measured in this run (fp64_peak)" if self.fp64_peak
                     else "37.2 TFLOP/s (profiles/r1_fp64_peak_ubench.json)",
                     note="FP64 tensor pipe (mma.sync f64; tcgen05 has no f64 kind); flops = the reference's operation "
                          "count (SURVEY §8d)", hbm_gbs_algorithmic=gbs)
        else:
            r.update(bound="hbm", achieved=gbs, peak=self.hbm_peak, unit="GB/s", frac=gbs / self.hbm_peak,
                     peak_source=self.hbm_src, fp64_tflops_algorithmic=tfs)
        return r

    # ---------------------------------------------------------------- Riccati configs (2, 5a-R, 5b-R)
    def run_riccati(self, cfg, steps, warmup, headline=False):
        torch = self.torch
        from lqr_b200 import _lib, ops, synthetic
        n, m, N, batch = cfg["n"], cfg["m"], cfg["N"], cfg["batch"]
        h = self.handle()
        L = _lib.riccati_layout(n, m, N)
        ldb = _lib.padded_batch(batch)
        kr = L.knot_count * L.rows_per_knot
        knots = torch.empty(ldb * kr, dtype=torch.float64, device="cuda")
        term = torch.empty(ldb * L.term_rows, dtype=torch.float64, device="cuda")
        Zp = torch.empty(ldb * L.z_rows, dtype=torch.float64, device="cuda")
        gains = torch.empty(ldb * L.gain_rows, dtype=torch.float64, device="cuda")
        info = torch.zeros(batch, dtype=torch.int32, device="cuda")
        per_inst = 8 * (kr + L.term_rows) * 2.2
        chunk = max(32, min(batch, int(1.5e9 / per_inst) // 32 * 32))
        prob_math, host_chunks = None, []
        for ci, first in enumerate(range(0, batch, chunk)):
            cnt = min(chunk, batch - first)
            seed = cfg["seed"] + 7919 * self.rank
            f = (synthetic.riccati_cartpole_chunk(cnt, seed, ci, N=N) if cfg["gen"] == "cartpole"
                 else synthetic.random_riccati_chunk(n, m, N, cnt, seed, ci))
            ops.riccati_pack(h, n, m, N, cnt, 0, *[f[k] for k in synthetic.RICCATI_NAMES],
                             knots[first * kr:], term[first * L.term_rows:])
            if ci == 0:
                prob_math = synthetic.riccati_to_math(f, 0, min(PARITY_INSTANCES, cnt))
            if headline:                # the e2e leg feeds the same instances from host memory
                host_chunks.append({k: f[k].cpu() for k in synthetic.RICCATI_NAMES})
            torch.cuda.synchronize()
            del f

        def step():
            ops.riccati_solve_packed(h, n, m, N, batch, 0, knots, term, Zp, gains, info)

        total_ms, per, launches, clocks = self.time_steps(h, step, steps, warmup)
        assert int(info.abs().max().item()) == 0, "numerical failure flagged in info[]"
        kernel = h.last_kernel
        if self.dumping():
            Zd = torch.empty(batch, L.z_rows, dtype=torch.float64, device="cuda")
            Kd = torch.empty(batch, N - 1, n, m, dtype=torch.float64, device="cuda")  # column-major m x n per knot
            kffd = torch.empty(batch, N - 1, m, dtype=torch.float64, device="cuda")
            ops.riccati_unpack(h, n, m, N, batch, Zp, gains, Zd, Kd, kffd)
            self.dump_outputs(cfg, dict(Z=Zd, K=Kd, kff=kffd, info=info))
            del Zd, Kd, kffd
        # parity of the timed output
        pc = prob_math["x0"].shape[0]
        Zd = torch.empty(pc, L.z_rows, dtype=torch.float64, device="cuda")
        ops.riccati_unpack(h, n, m, N, pc, Zp, None, Zd)
        torch.cuda.synchronize()
        parity = parity_riccati(prob_math, Zd.cpu().numpy(), n, m, N) if self.rank == 0 else None
        out = dict(total_ms=total_ms, per=per, launches=launches, clocks=clocks, kernel=kernel, parity=parity,
                   steps=steps, bytes_per=riccati_bytes(n, m, N), flops_per=riccati_flops(n, m, N))
        if headline:
            host = {k: torch.cat([c[k] for c in host_chunks]).pin_memory() for k in synthetic.RICCATI_NAMES}
            del host_chunks
            out["e2e"] = self.e2e_riccati(h, cfg, host, L)
        h.close()
        del knots, term, Zp, gains
        torch.cuda.empty_cache()
        return out

    def e2e_riccati(self, h, cfg, f, L):
        """End to end through lqrb_riccati_f64 with HOST pinned instance-major buffers (H2D + pack + solve + unpack +
        D2H in the timed region); also an LTI leg (the reference's actual LQRProblem form, src/lqr_problem.jl:1-11)."""
        torch = self.torch
        from lqr_b200 import _lib, ops, synthetic
        n, m, N, batch = cfg["n"], cfg["m"], cfg["N"], cfg["batch"]
        names = synthetic.RICCATI_NAMES
        host = f
        NN = L.z_rows
        Zh = torch.empty(batch, NN, dtype=torch.float64).pin_memory()
        infoh = torch.zeros(batch, dtype=torch.int32).pin_memory()

        def run(flags, src):
            ops.riccati(h, n, m, N, batch, flags, *[src[k] for k in names], Zh, None, None, infoh)

        def timed(flags, src):
            run(flags, src)
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(self.args.e2e_steps):
                run(flags, src)
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / self.args.e2e_steps

        e2e_s = timed(0, host)
        h2d = sum(host[k].numel() * 8 for k in names)
        d2h = Zh.numel() * 8 + infoh.numel() * 4
        # LTI: A, B, Q, R, q, r without the knot axis (knot 0 of every instance)
        lti = {k: (host[k][:, 0].contiguous().pin_memory() if k in ("A", "B", "Q", "R", "q", "r") else host[k])
               for k in names}
        lti_s = timed(_lib.FLAG_LTI, lti)
        lti_h2d = sum(lti[k].numel() * 8 for k in names)
        # the host->device link rate this rank sees while every rank copies at once (pinned source, one stream)
        dst = torch.empty_like(host["A"], device="cuda")
        dst.copy_(host["A"], non_blocking=True)
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            dst.copy_(host["A"], non_blocking=True)
        torch.cuda.synchronize()
        link_gbs = 3 * host["A"].numel() * 8 / (time.perf_counter() - t0) / 1e9
        return dict(e2e_s=e2e_s, h2d=h2d, d2h=d2h, lti_s=lti_s, lti_h2d=lti_h2d, link_gbs=link_gbs)

    # ---------------------------------------------------------------- KKT configs (3, 5a-K, 5b-K)
    def run_kkt(self, cfg, steps, warmup):
        torch = self.torch
        from lqr_b200 import _lib, ops, synthetic
        n, m, N, batch = cfg["n"], cfg["m"], cfg["N"], cfg["batch"]
        h = self.handle()
        p = np.zeros(N, dtype=np.int32)
        p[0] = p[-1] = n
        hm = _lib.HESS_BLOCKDIAG
        rows = _lib.kkt_data_rows(n, m, N, p, hm)
        NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
        ldb = _lib.padded_batch(batch)
        data = torch.empty(ldb * rows, dtype=torch.float64, device="cuda")
        dzp = torch.empty(ldb * NN, dtype=torch.float64, device="cuda")
        mp = torch.empty(ldb * P, dtype=torch.float64, device="cuda")
        info = torch.zeros(batch, dtype=torch.int32, device="cuda")
        chunk = max(32, min(batch, int(1.5e9 / (8 * rows * 2.6)) // 32 * 32))
        prob_math = None
        for ci, first in enumerate(range(0, batch, chunk)):
            cnt = min(chunk, batch - first)
            seed = cfg["seed"] + 7919 * self.rank
            f = (synthetic.dubins_kkt_chunk(cnt, seed, ci, N=N) if cfg["gen"] == "dubins"
                 else synthetic.random_kkt_chunk(n, m, N, cnt, seed, ci))
            ops.kkt_pack(h, n, m, N, cnt, p, hm, *[f[k] for k in synthetic.KKT_NAMES], data[first * rows:])
            if ci == 0:
                prob_math = synthetic.kkt_to_math(f, 0, min(PARITY_INSTANCES, cnt))
            torch.cuda.synchronize()
            del f

        def step():
            ops.kkt_solve_packed(h, n, m, N, batch, p, hm, False, 0, data, dzp, mp, None, info)

        total_ms, per, launches, clocks = self.time_steps(h, step, steps, warmup)
        assert int(info.abs().max().item()) == 0, "numerical failure flagged in info[]"
        kernel = h.last_kernel
        if self.dumping():
            dzd = torch.empty(batch, NN, dtype=torch.float64, device="cuda")
            multd = torch.empty(batch, P, dtype=torch.float64, device="cuda")
            ops.kkt_unpack(h, n, m, N, batch, p, hm, False, dzp, mp, None, dzd, multd, None)
            self.dump_outputs(cfg, dict(dz=dzd, mult=multd, info=info))
            del dzd, multd
        pc = prob_math["q"].shape[0]
        dz = torch.empty(pc, NN, dtype=torch.float64, device="cuda")
        mult = torch.empty(pc, P, dtype=torch.float64, device="cuda")
        ops.kkt_unpack(h, n, m, N, pc, p, hm, False, dzp, mp, None, dz, mult, None)
        torch.cuda.synchronize()
        parity = parity_kkt(prob_math, dz.cpu().numpy(), mult.cpu().numpy()) if self.rank == 0 else None
        h.close()
        del data, dzp, mp
        torch.cuda.empty_cache()
        return dict(total_ms=total_ms, per=per, launches=launches, clocks=clocks, kernel=kernel, parity=parity,
                    steps=steps, bytes_per=8 * (rows + NN + P), flops_per=kkt_flops(n, m, N, p))

    # ---------------------------------------------------------------- config 1: the reference's own single-instance case
    def run_fixture(self, cfg, steps, warmup):
        torch = self.torch
        from lqr_b200 import _lib, ops, problems
        h = self.handle()
        prob = problems.cartpole_fixture(cfg["N"])
        f = ops.kkt_flatten(prob)
        n, m, N = f["n"], f["m"], f["N"]
        p, hm = f["p"], f["hess_mode"]
        rows = _lib.kkt_data_rows(n, m, N, p, hm)
        NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
        dev = [None if f[k] is None else torch.from_numpy(np.ascontiguousarray(f[k])).cuda()
               for k in ("Q", "R", "Hux", "q", "r", "A", "B", "d", "D2", "C", "c")]
        data = torch.zeros(32 * rows, dtype=torch.float64, device="cuda")
        dzp = torch.zeros(32 * NN, dtype=torch.float64, device="cuda")
        mp = torch.zeros(32 * P, dtype=torch.float64, device="cuda")
        info = torch.zeros(1, dtype=torch.int32, device="cuda")
        ops.kkt_pack(h, n, m, N, 1, p, hm, *dev, data)

        def step():
            ops.kkt_solve_packed(h, n, m, N, 1, p, hm, False, 0, data, dzp, mp, None, info)

        total_ms, per, launches, clocks = self.time_steps(h, step, steps, warmup)
        kernel = h.last_kernel
        dz = torch.empty(1, NN, dtype=torch.float64, device="cuda")
        mult = torch.empty(1, P, dtype=torch.float64, device="cuda")
        ops.kkt_unpack(h, n, m, N, 1, p, hm, False, dzp, mp, None, dz, mult, None)
        torch.cuda.synchronize()
        if self.dumping():
            self.dump_outputs(cfg, dict(dz=dz, mult=mult, info=info))
        parity = parity_kkt(prob, dz.cpu().numpy(), mult.cpu().numpy()) if self.rank == 0 else None
        h.close()
        return dict(total_ms=total_ms, per=per, launches=launches, clocks=clocks, kernel=kernel, parity=parity,
                    steps=steps, bytes_per=8 * (rows + NN + P), flops_per=kkt_flops(n, m, N, p))

    # ---------------------------------------------------------------- config 4: Dubins SQP x 10
    def run_sqp(self, cfg, steps, warmup):
        torch = self.torch
        from lqr_b200 import _lib, ops, synthetic
        batch, N = cfg["batch"], cfg["N"]
        h = self.handle()
        Z0, x0, xf, o = synthetic.dubins_turn90_device(batch, cfg["seed"] + 7919 * self.rank, N=N)
        o = dict(o, iters=10, line_search=1)
        Z = Z0.clone()
        fp = torch.zeros(batch, dtype=torch.float64, device="cuda")
        fd = torch.zeros(batch, dtype=torch.float64, device="cuda")
        it = torch.zeros(batch, dtype=torch.int32, device="cuda")
        solves = [0]

        def step():
            Z.copy_(Z0)          # restart from the initial guess (a 0.5-GB device copy inside the timed region)
            solves[0] = ops.sqp_dubins(h, batch, o, x0, xf, Z, fp, fd, it)

        total_ms, per, launches, clocks = self.time_steps(h, step, steps, warmup)
        kernel = h.last_kernel
        if self.dumping():
            self.dump_outputs(cfg, dict(Z=Z, feas_p=fp, feas_d=fd, iters=it))
        conv = float(((fp < 1e-5) & (fd < 2e-5)).double().mean().item())
        parity = None
        if self.rank == 0:
            import oracle
            from oracle import sqp_dubins as S
            oracle.build()
            pc = PARITY_INSTANCES
            Zo, fpo, fdo, ito, _ = S.solve(Z0[:pc].cpu().numpy(), x0[:pc].cpu().numpy(), xf[:pc].cpu().numpy(), o)
            parity = dict(max_rel_err=_rel_rows(Z[:pc].cpu().numpy(), Zo), vs="oracle/sqp_dubins.py (numpy SQP loop "
                          "around the oracle KKT chain)", instances=pc,
                          iteration_counts_equal=bool(np.array_equal(it[:pc].cpu().numpy(), ito)),
                          converged_fraction=conv)
        n, m = 3, 2
        p = np.zeros(N, dtype=np.int32)
        p[0] = p[-1] = n
        rows = _lib.kkt_data_rows(n, m, N, p, _lib.HESS_BLOCKDIAG)
        NN, P = _lib.num_vars(n, m, N), _lib.num_cons(n, N, p)
        h.close()
        del Z, Z0
        torch.cuda.empty_cache()
        return dict(total_ms=total_ms, per=per, launches=launches, clocks=clocks, kernel=kernel, parity=parity,
                    steps=steps, units_per_step=solves[0], bytes_per=8 * (rows + NN + P),
                    flops_per=kkt_flops(n, m, N, p),
                    note="metric counts KKT solves (10 outer iterations + second-order-correction solves); roofline = "
                         "the packed-data KKT-solve HBM roofline of config 3 (the fused kernel linearises on the fly "
                         "and no longer moves those bytes)")


def entry_from(runner, cfg, r, world):
    """One `configs` entry from a run result (max over ranks of the timed region)."""
    (total_ms,) = runner.max_over_ranks(r["total_ms"])
    steps = r["steps"]
    ms = total_ms / steps
    units = r.get("units_per_step", cfg["batch"])
    kern_ms = statistics.mean(r["per"])
    e = {"key": cfg["key"], "baseline_config": cfg["baseline_config"], "workload": cfg["workload"],
         "n": cfg["n"], "m": cfg["m"], "N": cfg["N"], "batch_per_gpu": cfg["batch"], "n_gpus": world,
         "value": world * units / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
         "gpu_launches": int(r["launches"]), "kernel": r["kernel"], "clocks": r["clocks"],
         "roofline": runner.roofline(cfg, kern_ms, units, r["bytes_per"], r["flops_per"], r["kernel"], cfg["workload"]),
         "parity": r["parity"], "parity_tol": cfg["tol"]}
    if cfg["bound"] == "latency":
        e["roofline"]["bound"] = "latency"
        e["roofline"]["note"] = "single instance: a parity config, not a throughput config (SURVEY §8d)"
        e["latency_us"] = 1e3 * kern_ms
    if cfg["kind"] == "sqp":
        # the fused kernel linearises on the fly: restated bounds for what it actually has to move / compute per KKT solve
        N, n, m = cfg["N"], cfg["n"], cfg["m"]
        NN, P = N * n + (N - 1) * m, (N + 1) * n
        fused_bytes = 8 * (2 * NN + 2 * P)      # iterate in + out, kept multipliers in + out
        dfma = (runner.fp64_peak or {}).get("dfma_tflops") or 33.7
        tfs = r["flops_per"] * units / (kern_ms * 1e-3) / 1e12
        e["roofline"]["restated_for_fused_kernel"] = {
            "algorithmic_bytes_per_solve": fused_bytes,
            "hbm_frac": fused_bytes * units / (kern_ms * 1e-3) / 1e9 / runner.hbm_peak,
            "fp64_tflops": tfs, "fp64_frac_of_dfma_peak": tfs / dfma,
            "note": "with the linearisation fused the step is FP64-latency-bound, not HBM-bound: flops = the reference's "
                    "KKT operation count (linearisation not counted), peak = DFMA throughput measured in this run"}
    if r.get("note"):
        e["note"] = r["note"]
    if r["parity"] is not None:
        e["parity_ok"] = bool(r["parity"]["max_rel_err"] <= cfg["tol"])
    return e


# ------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--configs", default="all", help="comma list of config keys (c1,c2,c3,c4,5aR,5aK,5bR,5bK) or 'all'; "
                    "the headline c2 always runs")
    ap.add_argument("--batch-scale", type=float, default=1.0, help="scale every batch (debug only)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what each config's last timed step computed to DIR/<config key>_<name>.npy (float64, "
                         "a fixed seeded sample of instances, 60 MiB in all; rank 0's instances)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1 and args.impl == "ours":
        # convenience: re-launch ourselves under torchrun, one rank per GPU
        port = 29500 + os.getpid() % 2000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    want = [c["key"] for c in CONFIGS] if args.configs == "all" else [k for k in args.configs.split(",") if k]
    if HEADLINE not in want:
        want.insert(0, HEADLINE)
    cfgs = []
    for c in CONFIGS:
        if c["key"] in want:
            c = dict(c)
            if args.batch_scale != 1.0 and c["batch"] > 1:
                c["batch"] = max(32, int(c["batch"] * args.batch_scale) // 32 * 32)
            cfgs.append(c)
    head = next(c for c in cfgs if c["key"] == HEADLINE)
    n, m, N, batch = head["n"], head["m"], head["N"], head["batch"]
    config = {"workload": head["workload"], "n": n, "m": m, "N": N, "batch_per_gpu": batch,
              "global_batch": batch * max(1, args.gpus), "problem": "LTV affine LQR, Riccati backward pass + forward rollout",
              "l2": "inputs (2.1 GB per GPU) are far larger than the 126 MB L2; no explicit flush",
              "parallelism": f"batch slices over {args.gpus} GPU(s), no collective on the data path",
              "other_configs": [c["workload"] for c in cfgs if c["key"] != HEADLINE]}

    # ------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_time_config(head, target_seconds=60.0, steps=args.steps, warmup=args.warmup)
        config["reference_sample"] = r["sample"]
        others = []
        for c in cfgs:
            if c["key"] == HEADLINE:
                continue
            o = cpu_time_config(c, target_seconds=4.0)
            others.append({"key": c["key"], "workload": c["workload"], "value": o["value"], "unit": UNIT,
                           "ms_per_step": o["ms_per_step"], "cores": o["cores"], "sample": o["sample"], "kind": "port"})
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "configs": others,
                "note": "reference algorithm, C/OpenMP restatement (oracle/lqr_oracle.c) on a bounded sample of the "
                        "workload (see cpu_baseline.sample); LQR.jl is pure Julia and Julia is not installed in this image"}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------ our arm (GPU)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    runner = Runner(args, rank, local_rank, world)
    runner.dump_share = DUMP_BYTES // len(cfgs)
    fp64_peak = runner.measure_fp64_peak()

    entries, head_res = [], None
    for c in cfgs:
        is_head = c["key"] == HEADLINE
        t0 = time.perf_counter()
        if c["kind"] == "riccati":
            r = runner.run_riccati(c, args.steps, args.warmup, headline=is_head)
        elif c["kind"] == "kkt":
            r = runner.run_kkt(c, args.steps, args.warmup)
        elif c["kind"] == "fixture":
            r = runner.run_fixture(c, args.steps, args.warmup)
        else:
            r = runner.run_sqp(c, args.steps, args.warmup)
        e = entry_from(runner, c, r, world)
        e["wall_s"] = time.perf_counter() - t0
        entries.append(e)
        if is_head:
            head_res = (r, e)

    r, e = head_res
    e2e = r["e2e"]
    e2e_s, lti_s = runner.max_over_ranks(e2e["e2e_s"], e2e["lti_s"])
    if rank == 0:
        pcie_gbs = (e2e["h2d"] + e2e["d2h"]) / e2e_s / 1e9
        line = {
            "metric": METRIC, "value": e["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": e["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "e2e": {"value": world * batch / e2e_s, "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"],
                    "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": 1e3 * e2e_s,
                    "api": "lqrb_riccati_f64 (host pinned instance-major buffers)",
                    "pcie_gbs_per_gpu": pcie_gbs, "h2d_link_gbs_per_gpu": e2e["link_gbs"],
                    "h2d_frac_of_link": (e2e["h2d"] / e2e_s / 1e9) / e2e["link_gbs"],
                    "lti": {"value": world * batch / lti_s, "unit": UNIT, "ms_per_step": 1e3 * lti_s,
                            "h2d_bytes_per_step": e2e["lti_h2d"], "d2h_bytes_per_step": e2e["d2h"],
                            "what": "same call with LQRB_FLAG_LTI: one (A,B,Q,R,q,r) per instance, the reference's "
                                    "LQRProblem form (src/lqr_problem.jl:1-11); secondary number"}},
            "gpu_launches": e["gpu_launches"],
            "clocks": e["clocks"],
            "roofline": e["roofline"],
            "parity": e["parity"], "parity_tol": head["tol"], "parity_ok": e.get("parity_ok"),
            "fp64_peak": fp64_peak,
            "configs": entries,
            "all_parity_ok": all(x.get("parity_ok", True) for x in entries),
        }
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_time_config(head, target_seconds=12.0)
            line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": "port",
                                    "sample": cb["sample"], "sparse_kkt": sparse_leg(n, m, N, seed=0)}
            for x, c in zip(entries, cfgs):
                if c["key"] != HEADLINE:
                    o = cpu_time_config(c, target_seconds=3.0)
                    x["cpu_baseline"] = {"value": o["value"], "unit": UNIT, "cores": o["cores"], "kind": "port",
                                         "sample": o["sample"]}
        print(json.dumps(line))
    runner.sampler.stop()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
