"""The KKT kernels on the open-loop unstable inputs of tests/test_gpu_kkt_stability.py (tests/unstable_lqr.py).

  python tools/kkt_unstable_report.py [--kernel kkt_wp] [--share --chunks 16 --batch 1024]

Per family of the test file's default-dispatch cases (optionally those whose id contains --kernel): the largest
(error / rule) ratio, rule = max(1e-10, 4 x the C oracle's error against the refined solve), and the conditioning
estimate's bits (lqrb_kkt_last_condition) on the unstable and on the benign instances.  --share: the 5a-K shape
((12, 4), N = 1001, goal rows, kkt_hw), --chunks batches of --batch instances, half of them unstable: the estimate's
histogram, the share of instances re-solved by kkt_coop and the host-array call time with and without the re-solve
(kkt_refine = 1 / 0).  --no-refine: the family report on the tuned kernels' own output.  A batch is generated on the
host (1,024 instances at N = 1001 take about 3 GB), so the share of a large batch is measured chunk by chunk.  One JSON line per family and per share run on stdout.  Needs a GPU;
LQRB200_LIB selects another build of the library (lqr_b200/_lib.py)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def families(handle, kernel, refine):
    from tests import test_gpu_kkt_stability as T
    out = {}
    for c in T.CASES:
        if kernel and kernel not in c.id:
            continue
        fam, N, goal = c.values
        n, m, _, mid_p, hess, form, kern, opts, padded, tuned = fam
        prob, tr, eo = T._case(n, m, N, mid_p, hess, form, goal, T._seed(n, m, N, mid_p, hess, goal))
        padded = padded or (tuned and not goal)
        (dz, mult, info, _), name = T._solve(handle, prob, T._prefix(kern, goal, tuned), opts, padded)
        ratio = T.errors(dz, mult, tr) / T._rule(eo)
        f = out.setdefault(c.id.rsplit("-N", 1)[0], dict(ratio=0.0, worst="", info_ok=True, unstable=[], benign=[]))
        f["info_ok"] &= bool((info == 0).all())
        if ratio.max() > f["ratio"]:
            f["ratio"], f["worst"] = float(ratio.max()), f"N{N}-{'goal' if goal else 'free'}-i{int(ratio.argmax())}"
        if tuned and refine:  # (kkt_refine = 0 records no estimate)
            bits = handle.kkt_last_condition(T.B)[0]
            f["unstable"] += bits[0::2].tolist()
            f["benign"] += bits[1::2].tolist()
    for fid, f in out.items():
        for k in ("unstable", "benign"):
            v, cnt = np.unique(f[k], return_counts=True)
            f[k] = {int(a): int(b) for a, b in zip(v, cnt)}
        print(json.dumps(dict(family=fid, kkt_refine=refine, max_error_over_rule=round(f["ratio"], 3), at=f["worst"],
                              info_ok=f["info_ok"], bits_unstable=f["unstable"], bits_benign=f["benign"])), flush=True)


def share(handle, chunks, batch):
    from lqr_b200 import ops
    from tests.unstable_lqr import unstable_kkt
    hist_u, hist_b, resolved, t1, t0 = {}, {}, 0, 0.0, 0.0
    for c in range(chunks):
        prob = unstable_kkt(12, 4, 1001, batch, seed=77 + c)
        for refine in (1, 0):
            handle.set_option("kkt_refine", refine)
            if c == 0:
                ops.kkt_solve_problem(prob, handle=handle)  # warm-up
            t = time.perf_counter()
            ops.kkt_solve_problem(prob, handle=handle)
            dt = time.perf_counter() - t
            if refine:
                t1 += dt
                name = handle.last_kernel
                bits, r = handle.kkt_last_condition(batch)
                resolved += r
                for h, sl in ((hist_u, bits[0::2]), (hist_b, bits[1::2])):
                    for v in sl.tolist():
                        h[v] = h.get(v, 0) + 1
            else:
                t0 += dt
        handle.set_option("kkt_refine", 1)
        assert name.startswith("kkt_hw<12,4,"), name
    total = chunks * batch
    print(json.dumps(dict(shape="(12,4) N=1001 kkt_hw", instances=total, chunk=batch, resolved=int(resolved),
                          resolved_share=round(resolved / total, 4), bits_unstable=dict(sorted(hist_u.items())),
                          bits_benign=dict(sorted(hist_b.items())), host_call_s_refine=round(t1 / chunks, 3),
                          host_call_s_no_refine=round(t0 / chunks, 3))), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--kernel", default="", help="only the families whose case id contains this")
    ap.add_argument("--no-refine", action="store_true", help="kkt_refine = 0: the tuned kernels' own output")
    ap.add_argument("--share", action="store_true", help="measure the re-solve share on the 5a-K shape instead")
    ap.add_argument("--chunks", type=int, default=16)
    ap.add_argument("--batch", type=int, default=1024)
    a = ap.parse_args()
    import oracle
    from lqr_b200 import _lib
    oracle.build()
    h = _lib.Handle(0)
    try:
        if a.share:
            share(h, a.chunks, a.batch)
        else:
            h.set_option("kkt_refine", 0 if a.no_refine else 1)
            families(h, a.kernel, 0 if a.no_refine else 1)
    finally:
        h.close()


if __name__ == "__main__":
    main()
