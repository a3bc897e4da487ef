"""Solve time per right-hand side of k sequential pcg calls against one pcg_multi(k) call, and the V-cycle time per right-hand side,
on the BASELINE operators (one GPU, one part, AUTO formats), plus np.array_equal of every column of the multi call against the
single call at the timed size.

    python scripts/multi_rhs_sweep.py [--out profiles/r05_multi_rhs.json] [--reps 3] [--ks 1,2,4,8] [--small]

Per launch: pamg_time_kernel_multi(k) (one k-wide launch where the block's kernel has one) against k times pamg_time_kernel (the
single launch), CUDA events around each launch with the L2 flushed before it -- k sequential solves meet the matrix cold in every
launch, so a single launch with a cold L2 is the fair unit.  Kinds: 1 / 7 Jacobi sweep (+ r.z) and 6 SpMV + p.q of level-0 A, 2
residual A0 + restriction R0, 3 prolongation P0, 1 Jacobi sweep of level-1 A.

Times are device times (CUDA events, pamg_stats.solve_ms / vcycle_ms).  The sequential and the multi variant alternate within every
repeat, so drift of the shared machine hits both; the spread over repeats is recorded beside the median.  The card's name, power
limit and maximum SM clock are read once with a read-only nvidia-smi query and stored with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

LAUNCHES = [("A0 jacobi", 1, 0), ("A0 jacobi+dot", 7, 0), ("A0 mul+dot", 6, 0), ("A0 resid + R0 restrict", 2, 0),
            ("P0 add", 3, 0), ("A1 jacobi", 1, 1)]
WORKLOADS = [("poisson256", "poisson", (256, 256, 256)), ("elasticity96", "elasticity", (96, 96, 96)),
             ("jump256", "jump", (256, 256, 256))]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clock = [s.strip() for s in out[0].split(",")]
        return dict(name=name, power_limit=power, sm_clock_max=clock)
    except Exception as e:  # noqa: BLE001
        return dict(error=str(e))


def stats(v):
    v = np.asarray(v, dtype=float)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()), n=int(len(v)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_multi_rhs.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--small", action="store_true", help="32^3 / 12^3 sizes: a rehearsal of the script, not a measurement")
    args = ap.parse_args()
    from parallel_amg_b200 import _lib as L
    from util import det_vector

    ks = [int(k) for k in args.ks.split(",")]
    res = dict(card=card(), reps=args.reps, workloads={})
    for wname, kind, dims in WORKLOADS:
        if args.small:
            dims = (12, 12, 12) if kind == "elasticity" else (32, 32, 32)
        t0 = time.time()
        c = L.Context(1)
        if kind == "poisson":
            c.gallery_poisson(dims, (1, 1, 1))
        elif kind == "jump":
            c.gallery_diffusion_jump(dims, (1, 1, 1), blocks=8, kmax=1.0e4, eps_z=1.0e-3)
        else:
            c.gallery_elasticity(dims, (1, 1, 1))
        c.setup(c.default_options())
        c.set_rhs_capacity(max(ks))
        c.device_init()
        n = c.level_info(0, 0).n_own
        B = [[det_vector(n, seed=101 + j)] for j in range(max(ks))]
        w = dict(dims=list(dims), rows=int(n), setup_s=round(time.time() - t0, 1), k={})
        ref = [c.pcg(b, rtol=1e-8, maxiter=500) for b in B]  # warm-up and the reference bits
        w["iters"] = [r[1] for r in ref]
        w["launch_ms"] = {}
        for lname, kind, level in LAUNCHES:
            if level >= c.num_levels() - 1:
                continue
            one = float(np.median(c.time_kernel(kind, level, args.reps + 8, True)[3:]))
            row = dict(single=one)
            for k in ks:
                if k > 1:
                    mk = float(np.median(c.time_kernel_multi(k, kind, level, args.reps + 8, True)[3:]))
                    row[f"k{k}"] = mk
                    row[f"k{k}_vs_k_single"] = mk / (k * one)
            w["launch_ms"][lname] = row
            print(wname, lname, json.dumps(row), flush=True)
        for k in ks:
            got = c.pcg_multi(B[:k], rtol=1e-8, maxiter=500, mode=1)  # warm-up (graph capture) and the bit check
            equal = all(np.array_equal(g[0][0], r[0][0]) and g[1] == r[1] and np.array_equal(g[2], r[2]) for g, r in zip(got, ref))
            names = c.trace_names()
            seq, mul, vseq, vmul = [], [], [], []
            c.vcycle(B[0])
            c.vcycle_multi(B[:k])
            for _ in range(args.reps):
                t = 0.0
                for j in range(k):
                    c.pcg(B[j], rtol=1e-8, maxiter=500)
                    t += c.stats().solve_ms
                seq.append(t / k)
                c.pcg_multi(B[:k], rtol=1e-8, maxiter=500, mode=1)
                mul.append(c.stats().solve_ms / k)
                c.vcycle(B[0])
                vseq.append(c.stats().vcycle_ms)
                c.vcycle_multi(B[:k])
                vmul.append(c.stats().vcycle_ms / k)
            w["k"][str(k)] = dict(bit_identical=bool(equal), pcg_ms_per_rhs_sequential=stats(seq), pcg_ms_per_rhs_multi=stats(mul),
                                  speedup_per_rhs=float(np.median(seq) / np.median(mul)), vcycle_ms_per_rhs_single=stats(vseq),
                                  vcycle_ms_per_rhs_multi=stats(vmul), k_wide_launches=[s for s in names if f" x" in s][:12])
            print(wname, k, json.dumps(w["k"][str(k)], default=str)[:400], flush=True)
        res["workloads"][wname] = w
        del c
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
