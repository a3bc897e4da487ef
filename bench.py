#!/usr/bin/env python
"""bench.py — AMG-PCG solve throughput (DOF/s) on N B200s, plus roofline / CPU baseline / e2e / parity record.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload poisson3d-256|poisson3d-128|...]
  python bench.py --impl reference ...     # the CPU oracle port timed on the host cores

A "step" is one whole AMG-preconditioned CG solve (x0 = 0, b = A*xstar, to ||r|| <= 1e-8 ||r0||) of
BASELINE.json configs[2] (3-D Poisson 7-point 256^3, strong-scaled over N = 1/2/4/8 GPUs as
(1,1,1)/(2,1,1)/(2,2,1)/(2,2,2) Cartesian blocks).  The hierarchy is built on the host and uploaded
once (outside the timed region, as the north star prescribes).  `value` times K solves with b
resident in HBM (CUDA events inside the library, max over ranks); `e2e` times the same solves
through the C-ABI call pamg_pcg with pinned HOST buffers (H2D of b, D2H of x inside the region).

Parity record (every N): the iteration count and residual history of the timed solve are ASSERTED equal to the
C oracle's on the same hierarchy and right-hand side (`parity.iters_match`), and a small problem (40^3) is run on
the same N ranks -- one part per GPU, fused halo roles, CUDA-IPC peer memory: the production multi-GPU path -- against
the oracle's N-part V-cycle and PCG (`parity.small`: vcycle_rel_err <= 1e-12, identical iterations).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    "poisson3d-256": dict(dims=(256, 256, 256), desc="3D Poisson 7-point 256^3 (16.7M DOF), b=A*xstar, x0=0, rtol 1e-8"),
    "poisson3d-128": dict(dims=(128, 128, 128), desc="3D Poisson 7-point 128^3 (2.1M DOF), b=A*xstar, x0=0, rtol 1e-8"),
    "poisson3d-64": dict(dims=(64, 64, 64), desc="3D Poisson 7-point 64^3 (262k DOF), b=A*xstar, x0=0, rtol 1e-8"),
    # BASELINE.json configs[3]: 27-point node stencil, 3 DOFs per node, rigid-body near-nullspace SA
    "elasticity3d-96": dict(dims=(96, 96, 96), kind="elasticity",
                            desc="3D linear elasticity Q1, 96^3 nodes x 3 DOF (2.65M DOF), rigid-body SA, b=A*xstar, x0=0, rtol 1e-8"),
    # BASELINE.json configs[4] (512^3 on 8 GPUs) and reduced sizes of the same operator: -div(K grad u), K = diag(k,k,1e-3 k),
    # k in {1, 1e4} on an 8^3 checkerboard; strength threshold 0.08 (without it PCG needs > 400 iterations)
    "diffusion-jump-3d-512": dict(dims=(512, 512, 512), kind="jump", opts=dict(eps_strength=0.08),
                                  desc="3D jump-coefficient anisotropic diffusion 512^3 (134M DOF), eps 0.08, b=A*xstar, x0=0, rtol 1e-8"),
    "diffusion-jump-3d-256": dict(dims=(256, 256, 256), kind="jump", opts=dict(eps_strength=0.08),
                                  desc="3D jump-coefficient anisotropic diffusion 256^3 (16.7M DOF), eps 0.08, b=A*xstar, x0=0, rtol 1e-8"),
    "diffusion-jump-3d-128": dict(dims=(128, 128, 128), kind="jump", opts=dict(eps_strength=0.08),
                                  desc="3D jump-coefficient anisotropic diffusion 128^3 (2.1M DOF), eps 0.08, b=A*xstar, x0=0, rtol 1e-8"),
    "elasticity3d-48": dict(dims=(48, 48, 48), kind="elasticity",
                            desc="3D linear elasticity Q1, 48^3 nodes x 3 DOF (332k DOF), rigid-body SA, b=A*xstar, x0=0, rtol 1e-8"),
}
PARTS = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}
RTOL, MAXITER = 1e-8, 200
SMOOTHER_DESC = "jacobi(2/3) 1+1"
# the other BASELINE.json configs, measured after the headline workload: N = 1 -> configs[1] and configs[3], N = 8 -> configs[4]
SECONDARY = {1: ("poisson3d-128", "elasticity3d-96"), 8: ("diffusion-jump-3d-512",)}


def make_problem(c, wl, nparts):
    if wl.get("kind") == "elasticity":
        c.gallery_elasticity(wl["dims"], PARTS[nparts])
    elif wl.get("kind") == "jump":
        c.gallery_diffusion_jump(wl["dims"], PARTS[nparts], blocks=8, kmax=1.0e4, eps_z=1.0e-3)
    else:
        c.gallery_poisson(wl["dims"], PARTS[nparts])


def xstar(n):
    """Known solution of the benchmark system: deterministic pseudo-random values in (-1, 1)
    (multiplicative hash of the gid, identical bits everywhere).  SURVEY.md 8d proposed b = A*1, but
    that right-hand side is degenerate for this hierarchy (PCG converges in ONE iteration at 32^3 and
    128^3), so it would not measure a solve; see DESIGN.md "Benchmark right-hand side"."""
    i = np.arange(n, dtype=np.uint64)
    return ((i * np.uint64(2654435761) + np.uint64(40503)) % np.uint64(2 ** 32)).astype(np.float64) / 2.0 ** 31 - 1.0


DUMP_MAX_ENTRIES = 1 << 21   # solution entries --dump-outputs writes: 16 MB of values + 16 MB of indices


def dump_outputs(out_dir, x, it, hist):
    """--dump-outputs: what a caller of the timed solve receives from its last step, as float64 .npy files -- the solution
    (x.npy at the global indices x_index.npy: all of it, or a fixed seeded sample of DUMP_MAX_ENTRIES entries when larger),
    the residual history (||r_k||, k = 0 .. iters) and the iteration count -- so that two builds can be compared output
    for output on identical inputs."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(x)
    idx = np.arange(n) if n <= DUMP_MAX_ENTRIES else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ENTRIES, replace=False))
    np.save(os.path.join(out_dir, "x.npy"), np.asarray(x, np.float64)[idx])
    np.save(os.path.join(out_dir, "x_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "residual_history.npy"), np.asarray(hist, np.float64))
    np.save(os.path.join(out_dir, "iters.npy"), np.array([it], np.float64))


def config_of(workload, wl, nparts, iters, levels):
    """Identical key set (and, by the asserted parity, identical values) in both arms."""
    return dict(workload=workload, description=wl["desc"], parts=list(PARTS[nparts]), iters=int(iters), levels=int(levels),
                smoother=SMOOTHER_DESC, rtol=RTOL)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload, n_gpus):
    """dram__bytes_read + dram__bytes_write per launch of the roofline kernel from a committed `ncu --set full` capture
    of THIS workload at THIS number of GPUs (profiles/ncu_traffic.json), else None -- never a number from another case."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            return json.load(fh).get(workload, {}).get(str(n_gpus), {}).get("spmv_A0_dram_bytes_per_launch")
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    power_w_max=max(pw) if pw else None, samples=len(sm), reasons=sorted(reasons))


def cpu_solve_timed(c, nparts, b_parts, reps, threads=None):
    """The oracle's C/OpenMP solve phase on the host cores, same hierarchy (copied out through the C ABI), same rhs."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    from parallel_amg_b200 import _lib as L
    L.set_num_threads(threads or os.cpu_count() or 1)   # launchers export OMP_NUM_THREADS=1; the oracle shares the process's OpenMP runtime
    co = c_oracle.COracle.from_product_context(c, nparts)
    times, it, hist, x = [], 0, None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        x, it, hist = co.pcg(b_parts, RTOL, MAXITER, True)
        times.append(time.perf_counter() - t0)
    co.close()
    return times, it, hist, x


def other_krylov_drivers(c, nparts, b_parts, own_all, b):
    """SURVEY 8(f3) record: flexible CG and restarted flexible GMRES through the C ABI on this workload, each against the C
    oracle's restatement of the same driver (iterations and residual history).  Returns a dict; never raises."""
    out = {}
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import c_oracle
        co = c_oracle.COracle.from_product_context(c, nparts)
        rhs = [b[o] for o in own_all]
        for name, dev, ref in (("fcg", lambda: c.fcg(b_parts, RTOL, MAXITER), lambda: co.pcg(rhs, RTOL, MAXITER, True, flexible=True)),
                               ("fgmres30", lambda: c.fgmres(b_parts, RTOL, MAXITER, 30, True), lambda: co.fgmres(rhs, RTOL, MAXITER, 30, True))):
            try:
                dev()                                   # warm-up (graph capture, basis allocation)
                x, it, hist, ok = dev()
                ms = c.stats().solve_ms
                xr, it_ref, hist_ref = ref()
                out[name] = dict(iters=int(it), oracle_iters=int(it_ref), iters_match=bool(it == it_ref), converged=bool(ok),
                                 history_match=bool(len(hist) == len(hist_ref) and np.allclose(hist, hist_ref, rtol=1e-7)),
                                 device_ms=float(ms))
            except Exception as e:  # noqa: BLE001
                out[name] = dict(error=f"{type(e).__name__}: {e}")
        co.close()
    except Exception as e:  # noqa: BLE001
        out["error"] = f"{type(e).__name__}: {e}"
    return out


def write_trace(c, part, path):
    """Per-kernel timeline of one resident solve: start-to-start deltas (device globaltimer) of every kernel
    of a PCG iteration, median over the iterations.  Diagnostic only (not part of any reported number)."""
    c.trace_enable(1 << 16)
    it, hist, ok = c.pcg_resident(RTOL, MAXITER, True)
    t = c.trace_read(part).astype(np.int64)
    c.trace_enable(0)
    names = c.trace_names()
    k = len(names)
    head = len(t) - it * k if k else 0      # k_pcg_init (+ k_check when the check is not folded into it) precede the iterations
    body = t[max(head, 0):]
    nit = min(it, len(body) // k) if k else 0
    with open(path, "w") as fh:
        fh.write(f"# iterations {it}, kernels per iteration {k}, records {len(t)}\n")
        if nit < 2:
            return
        d = np.diff(body[: nit * k + 1].astype(np.float64))[: (nit - 1) * k + k - 1]
        d = np.concatenate([d, [np.nan] * (nit * k - len(d))]).reshape(nit, k)
        med = np.nanmedian(d, axis=0) / 1e3
        fh.write(f"# median start-to-start delta per kernel (us); sum = {np.nansum(med):.1f} us per iteration\n")
        for nm, m in zip(names, med):
            fh.write(f"{m:9.2f}  {nm}\n")


def small_parity(rank, world, local_rank, nparts):
    """40^3 Poisson on the same N ranks (one part per GPU, CUDA-IPC peer memory, fused halo roles) against the oracle's
    N-part V-cycle / PCG on the same operators, twice: with AUTO formats (CSR-stream at this size, everything below level 0
    in the fused replicated tail) and with SELL-C-sigma forced and the coarse levels kept distributed (tail_rows = 600), i.e.
    the kernel family and halo roles the 256^3 production run uses.  Returns the record on every rank (max over ranks)."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    from parallel_amg_b200 import _lib as L
    from parallel_amg_b200.distributed import connect_parts
    dims = (40, 40, 40)
    L.set_num_threads(max(1, (os.cpu_count() or 1) // max(world, 1)))
    rec = dict(problem="poisson3d-40", n_parts=nparts, tol_vcycle=1e-12, vcycle_rel_err=0.0, solution_max_abs_err=0.0, iters_match=True,
               variants=[])
    for vname, kopts in (("auto", {}), ("sell-distributed", dict(spmv_format=L.FORMAT_SELL, tail_rows=600))):
        c = L.Context(nparts)
        c.gallery_poisson(dims, PARTS[nparts])
        c.setup(c.default_options(**kopts))
        if world > 1:
            connect_parts(c, rank, world, local_rank)
        else:
            c.device_init([0], [local_rank])
        co = c_oracle.COracle.from_product_context(c, nparts)
        n, _ = c.global_size()
        own = [c.index_maps(0, p)[0] for p in range(nparts)]
        me = rank if world > 1 else 0
        v = xstar(n)[::-1].copy()
        z_ref = co.vcycle([v[o] for o in own])
        z = c.vcycle([v[own[p]] if p == me else None for p in range(nparts)])
        scale = max(float(np.abs(r).max()) for r in z_ref)
        err = float(np.abs(z[me] - z_ref[me]).max()) / scale
        rhs = c.host_matvec_global(xstar(n))
        x_ref, it_ref, hist_ref = co.pcg([rhs[o] for o in own], RTOL, MAXITER, True)
        x, it, hist, ok = c.pcg([rhs[own[p]] if p == me else None for p in range(nparts)], RTOL, MAXITER, True)
        match = bool(ok and it == it_ref and len(hist) == len(hist_ref) and np.allclose(hist, hist_ref, rtol=1e-7))
        xerr = float(np.abs(x[me] - x_ref[me]).max())
        stt = c.stats()
        if world > 1:
            t = torch.tensor([err, xerr, 0.0 if match else 1.0], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            err, xerr, bad = [float(a) for a in t.cpu()]
            match = bad == 0.0
            dist.barrier()
        rec["variants"].append(dict(name=vname, vcycle_rel_err=err, iters=int(it), oracle_iters=int(it_ref), iters_match=match,
                                    solution_max_abs_err=xerr, fused_halo=int(stt.fused_halo), tail_level=int(stt.tail_level),
                                    format_A0=int(stt.format[0])))
        rec["vcycle_rel_err"] = max(rec["vcycle_rel_err"], err)
        rec["solution_max_abs_err"] = max(rec["solution_max_abs_err"], xerr)
        rec["iters_match"] = bool(rec["iters_match"] and match)
        co.close()
        c.close()
    return rec


def measure(workload, args, rank, world, local_rank, steps, warmup, headline):
    """One workload on the N ranks: setup, resident solves (value), C-ABI solves with host buffers (e2e), kernel timings,
    parity of the timed solve against the C oracle.  Returns the record on rank 0 (None elsewhere)."""
    import torch
    import torch.distributed as dist
    from parallel_amg_b200 import _lib as L
    wl = WORKLOADS[workload]
    nparts = args.gpus
    dims = wl["dims"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Host setup: rank 0 builds the hierarchy once with every host core and hands it to the other ranks through a
    # shared-memory file (each loads only its own part in full); --replicate-setup repeats it in every rank instead.
    share = world > 1 and not args.replicate_setup
    L.set_num_threads((os.cpu_count() or 1) if share else max(1, (os.cpu_count() or 1) // max(world, 1)))  # torchrun exports OMP_NUM_THREADS=1
    c = L.Context(nparts)
    t0 = time.perf_counter()
    opts_kw = wl.get("opts", {})
    if share:
        from parallel_amg_b200.distributed import shared_setup
        need_bytes = 400 * int(np.prod(dims)) * (12 if wl.get("kind") == "elasticity" else 1)   # generous file-size estimate

        def build(ctx):
            make_problem(ctx, wl, nparts)
            ctx.setup(ctx.default_options(**opts_kw))

        n, nnz = shared_setup(c, build, rank, world, tag=workload, need_bytes=need_bytes)
    else:
        make_problem(c, wl, nparts)
        if world > 1:  # replicated setup in waves so that the box's memory holds the concurrent copies
            try:
                avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) * 1024
            except Exception:
                avail = 64 << 30
            need = 1000 * int(np.prod(dims)) * (30 if wl.get("kind") == "elasticity" else 1)  # bytes, generous
            per_wave = max(1, min(world, int(0.6 * avail // need)))
            for w0 in range(0, world, per_wave):
                if w0 <= rank < w0 + per_wave:
                    c.setup(c.default_options(**opts_kw))
                dist.barrier()
        else:
            c.setup(c.default_options(**opts_kw))
        n, nnz = c.global_size()
    setup_s = time.perf_counter() - t0
    if world > 1:
        from parallel_amg_b200.distributed import connect_parts
        connect_parts(c, rank, world, local_rank)
        mine = [rank]
    else:
        c.device_init([0], [local_rank])
        mine = [0]
    have_A = (not share) or rank == 0      # only the rank that ran the gallery holds the global matrix
    xs_true = xstar(n)
    if share:  # b = A x* is computed where A lives and broadcast through the GPUs
        tb = torch.from_numpy(c.host_matvec_global(xs_true)).cuda() if rank == 0 else torch.empty(n, dtype=torch.float64, device="cuda")
        dist.broadcast(tb, src=0)
        b = tb.cpu().numpy()
        del tb
    else:
        b = c.host_matvec_global(xs_true)
    own = {p: c.index_maps(0, p)[0] for p in mine}
    # pinned host buffers for the e2e leg (the library copies from/to these pointers)
    b_pin = {p: torch.from_numpy(b[own[p]].copy()).pin_memory() for p in mine}
    b_parts = [b_pin[p].numpy() if p in b_pin else None for p in range(nparts)]
    x_pin = {p: torch.empty(len(own[p]), dtype=torch.float64).pin_memory() for p in mine}
    x_parts = [x_pin[p].numpy() if p in x_pin else None for p in range(nparts)]

    # ---- value: K solves with b resident in HBM ---------------------------------------------
    c.load_rhs(b_parts)
    for _ in range(warmup):
        it, hist, ok = c.pcg_resident(RTOL, MAXITER, True)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0 and headline:
        sampler.start()
    dev_ms, launches = 0.0, 0
    t_wall = time.perf_counter()
    for _ in range(steps):
        it, hist, ok = c.pcg_resident(RTOL, MAXITER, True)
        st = c.stats()
        dev_ms += st.solve_ms
        launches += st.kernel_launches
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t_wall)
    clocks = sampler.stop() if rank == 0 and headline else None
    assert ok, "PCG did not converge"
    x = c.read_solution()
    # true-residual check of the timed result (size-independent property): ||b - A x|| <= rtol ||b||
    xg = np.zeros(n)
    for p in mine:
        xg[own[p]] = x[p]
    if world > 1:
        t = torch.from_numpy(xg).cuda()
        dist.all_reduce(t)
        xg = t.cpu().numpy()
    true_rel = float(np.linalg.norm(b - c.host_matvec_global(xg)) / np.linalg.norm(b)) if have_A else 0.0
    assert true_rel <= 2e-8, f"true residual {true_rel}"
    sol_err = float(np.abs(xg - xs_true).max())
    if args.dump_outputs and headline and rank == 0:
        dump_outputs(args.dump_outputs, xg, it, hist)

    if args.trace and headline:
        write_trace(c, mine[0], args.trace + f".rank{rank}.txt")

    # ---- e2e: the C-ABI call with host buffers (H2D b, D2H x inside the timed region) ---------
    for _ in range(2):
        c.pcg(b_parts, RTOL, MAXITER, True, out=x_parts)
    barrier()
    t_e2e = time.perf_counter()
    for _ in range(steps):
        xh, it2, hist2, ok2 = c.pcg(b_parts, RTOL, MAXITER, True, out=x_parts)
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t_e2e)

    # ---- V-cycle ms and per-kernel roofline (CUDA events on the library's stream) --------------
    vc = c.time_kernel(5, 0, 23, False)[3:]
    kern = {}
    info = c.level_info(0, mine[0])
    n_own, nnz_oo = info.n_own, info.nnz[0]
    stt = c.stats()
    # SURVEY 8(d) bytes of a CSR SpMV with fp64 values (12 B per entry + row pointers + x + y) ...
    csr_bytes = 12 * nnz_oo + 4 * (n_own + 1) + 8 * n_own + 8 * n_own
    # ... and what the kernel that runs has to move: a value-indexed SELL block (DESIGN 4.1b: <= 255 distinct values -> int32 column +
    # one byte per entry, no row pointers) moves 5 B per entry.  The roofline fraction is taken on the bytes of the format that runs;
    # the fp64-CSR-equivalent rate is reported beside it.
    vi_a0 = bool(stt.value_indexed[0] & 1)
    vi_wide = bool(stt.value_indexed[0] & 8)        # two index bytes (256 .. 4095 distinct values)
    spmv_bytes = ((6 if vi_wide else 5) * nnz_oo + 16 * n_own) if vi_a0 else csr_bytes
    algo = {0: ("spmv A0", spmv_bytes, csr_bytes), 1: ("jacobi sweep A0", spmv_bytes + 16 * n_own, csr_bytes + 16 * n_own)}
    for kind, (name, nbytes, eq) in algo.items():
        ms = c.time_kernel(kind, 0, 13, True)[3:]
        kern[name] = dict(ms=float(np.mean(ms)), gbs=nbytes / (float(np.mean(ms)) * 1e-3) / 1e9, bytes=int(nbytes),
                          fp64_csr_equivalent_gbs=eq / (float(np.mean(ms)) * 1e-3) / 1e9, fp64_csr_equivalent_bytes=int(eq))
    kname = {L.FORMAT_SELL: (f"k_spmv_sell_vi4<MUL> (value-indexed SELL-C-sigma: int32 column + {2 if vi_wide else 1} byte(s) into a dictionary of the distinct fp64 "
                             "values, C=128, 128-bit column loads, 4 interleaved rows per lane, persistent CTAs)") if vi_a0 else
             "k_spmv_sell<RPT=2,MUL> (SELL-C-sigma, C=64, 128-bit value loads, persistent CTAs)",
             L.FORMAT_STREAM: "k_spmv_stream<MUL> (CSR-stream, 128-bit coalesced loads, smem-staged products)"}.get(
                 stt.format[0], f"k_spmv<lanes={stt.lanes[0]},MUL> (sub-warp CSR)")

    if world > 1:
        t = torch.tensor([dev_ms, wall_ms, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, e2e_ms = [float(v) for v in t.cpu()]
        tl = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(tl)
        launches = int(tl.item())

    # While rank 0 runs the CPU oracle the other ranks must SLEEP: ranks spinning in an NCCL barrier take a core each and
    # an oversubscribed OpenMP team is an order of magnitude slower (measured: 40 s instead of 3 s per solve on 8 ranks).
    flag = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp",
                        f"pamg_bench_{os.environ.get('MASTER_PORT', '0')}_{workload}_{args.gpus}.cpu_done")
    if world > 1:
        if rank == 0 and os.path.exists(flag):
            os.remove(flag)
        barrier()
    rec = None
    if rank == 0:
        try:
            # ---- the same solve on the host cores by the C oracle: CPU baseline AND parity of the timed solve ---------
            cpu = None
            parity = dict(iters=int(it), oracle_iters=None, iters_match=None, history_match=None)
            if not args.no_cpu_baseline and n <= 40_000_000:   # the 512^3 secondary would copy 37 GB of hierarchy for the oracle
                own_all = [c.index_maps(0, p)[0] for p in range(nparts)]
                reps = args.cpu_reps if headline else 1
                cores = max(1, (os.cpu_count() or 1) - (world - 1))   # the sleeping ranks still own a helper thread each
                times, it_cpu, hist_cpu, _ = cpu_solve_timed(c, nparts, [b[o] for o in own_all], reps, threads=cores)
                cpu = dict(value=n / min(times), unit="DOF/s", cores=cores, kind="port",
                           sample=f"{reps} whole solve(s) ({it_cpu} iterations each) of the same workload on the same {nparts}-part hierarchy, best one; "
                                  f"C/OpenMP oracle port on {cores} host threads (no reference code exists)",
                           seconds=[round(t, 3) for t in times], iters=int(it_cpu))
                hmatch = bool(len(hist) == len(hist_cpu) and np.allclose(hist, hist_cpu, rtol=1e-7))
                parity = dict(iters=int(it), oracle_iters=int(it_cpu), iters_match=bool(it == it_cpu), history_match=hmatch)
                assert it == it_cpu, f"PCG iterations differ from the C oracle: device {it}, oracle {it_cpu}"
                assert hmatch, "PCG residual history differs from the C oracle's beyond 1e-7 relative"
            peak, peak_src = peaks()
            dom = kern["spmv A0"]
            rec = dict(
                value=n * steps / (dev_ms * 1e-3), ms_per_step=dev_ms / steps, n=int(n), iters=int(it), levels=c.num_levels(),
                vcycle_ms=float(np.mean(vc)), wall_ms_per_step=wall_ms / steps, true_residual_rel=true_rel, solution_max_err=sol_err,
                roofline=dict(bound="hbm", kernel=kname + " level 0: y = A x, fp64 arithmetic / int32 columns", achieved=dom["gbs"],
                              peak=peak, unit="GB/s", frac=dom["gbs"] / peak, peak_source=peak_src, traffic=ncu_traffic(workload, args.gpus),
                              algorithmic_bytes_per_launch=dom["bytes"], ms_per_launch=dom["ms"],
                              frac_of_nominal_8TBs=dom["gbs"] / 8000.0, value_indexed=vi_a0, index_bytes=(2 if vi_wide else 1) if vi_a0 else 0,
                              fp64_csr_equivalent=dict(bytes_per_launch=dom["fp64_csr_equivalent_bytes"], gbs=dom["fp64_csr_equivalent_gbs"],
                                                       frac=dom["fp64_csr_equivalent_gbs"] / peak,
                                                       note="SURVEY 8(d) bytes of the same product with 12 B per entry; > 1 means fewer bytes cross the pins than a CSR fp64 kernel needs")),
                kernels=kern,
                e2e=dict(value=n * steps / (e2e_ms * 1e-3), unit="DOF/s", h2d_bytes_per_step=8 * n, d2h_bytes_per_step=8 * n,
                         ms_per_step=e2e_ms / steps),
                gpu_launches=int(launches), clocks=clocks, cpu_baseline=cpu, parity=parity,
                host_setup_s=round(setup_s, 1), host_setup="rank 0 + shared-memory hand-off" if share else "every rank")
            if world == 1 and not headline and n <= 3_000_000 and not args.no_cpu_baseline and wl.get("kind") is None:
                rec["krylov"] = other_krylov_drivers(c, nparts, b_parts, [c.index_maps(0, p)[0] for p in range(nparts)], b)
        finally:   # whatever happens here, the sleeping ranks must be released
            if world > 1:
                open(flag, "w").close()
    elif world > 1:
        while not os.path.exists(flag):
            time.sleep(0.05)
    barrier()
    if world > 1 and rank == 0:
        os.remove(flag)
    c.close()
    return rec


def run_reference(args, wl, rank, world):
    """--impl reference: there is no reference code to run (SURVEY.md 0) and no Julia; the arm times
    the CPU oracle port (oracle/pamg_oracle.c) with all host threads on the same config."""
    if rank != 0:
        return
    from parallel_amg_b200 import _lib as L
    nparts = args.gpus
    L.set_num_threads(os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)  # the C oracle uses every host core
    c = L.Context(nparts)
    make_problem(c, wl, nparts)
    c.setup(c.default_options(**wl.get("opts", {})))
    n, nnz = c.global_size()
    b = c.host_matvec_global(xstar(n))
    own = [c.index_maps(0, p)[0] for p in range(nparts)]
    b_parts = [b[o] for o in own]
    times, it, hist, x = cpu_solve_timed(c, nparts, b_parts, args.warmup + args.steps)
    if args.dump_outputs:
        xg = np.zeros(n)
        for o, xp in zip(own, x):
            xg[o] = xp
        dump_outputs(args.dump_outputs, xg, it, hist)
    timed = times[args.warmup:]
    total = float(sum(timed))
    cores = os.cpu_count()
    val = n * len(timed) / total
    line = dict(impl="reference", metric="amg_pcg_solve_dof_per_s", value=val, unit="DOF/s", n_gpus=args.gpus, steps=len(timed),
                warmup=args.warmup, ms_per_step=1e3 * total / len(timed), higher_is_better=True, scaling="strong",
                vs_baseline=None, dtype="f64", data="synthetic",
                config=config_of(args.workload, wl, nparts, it, c.num_levels()),
                note="no reference code exists (README+LICENSE only) and Julia is absent: this is the repo's C/OpenMP "
                     "oracle port of the same algorithm on the same hierarchy (built by the host setup, bit-exact vs the "
                     "oracle setup in tests)",
                cpu_baseline=dict(value=val, unit="DOF/s", cores=cores, kind="port", sample="whole solve, every step",
                                  omp_threads=int(os.environ.get("OMP_NUM_THREADS", cores))),
                e2e=dict(value=val, unit="DOF/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="poisson3d-256", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the C-oracle solve (CPU baseline and iteration parity of the timed solve)")
    ap.add_argument("--cpu-reps", type=int, default=3, help="whole CPU solves timed for cpu_baseline (best one is reported)")
    ap.add_argument("--secondary", default="auto", help="'auto': the other BASELINE configs that fit this N (see SECONDARY), 'none', or a comma list of workloads")
    ap.add_argument("--no-small-parity", action="store_true")
    ap.add_argument("--smoother", default="jacobi")
    ap.add_argument("--replicate-setup", action="store_true", help="N > 1: every rank runs the host setup itself (default: rank 0 builds, the others load it from shared memory)")
    ap.add_argument("--trace", default=None, help="write a per-kernel timeline of one solve (device globaltimer) to this file prefix")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the solution (sampled above 2M entries), residual history and iteration count of the last timed solve "
                         "as float64 .npy files into DIR")
    args = ap.parse_args()
    if args.gpus not in PARTS:
        raise SystemExit("--gpus must be 1, 2, 4 or 8")
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return
    if world != args.gpus and not (world == 1 and args.gpus == 1):
        raise SystemExit(f"WORLD_SIZE={world} but --gpus {args.gpus}: launch with torchrun --nproc-per-node {args.gpus}")
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the product path has no CPU fallback (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    rec = measure(args.workload, args, rank, world, local_rank, args.steps, args.warmup, headline=True)
    small = None if args.no_small_parity else small_parity(rank, world, local_rank, args.gpus)

    # the other BASELINE.json configs that fit this N: a driver-visible record, never allowed to fail the headline line
    if args.secondary == "auto":
        names = SECONDARY.get(args.gpus, ()) if args.workload == "poisson3d-256" else ()
    elif args.secondary in ("none", ""):
        names = ()
    else:
        names = tuple(s for s in args.secondary.split(",") if s)
    secondary = {}
    for name in names:
        ok_local = 1.0
        try:
            r2 = measure(name, args, rank, world, local_rank, min(args.steps, 5), 3, headline=False)
        except Exception as e:  # noqa: BLE001
            r2, ok_local = dict(error=f"{type(e).__name__}: {e}"[:300]), 0.0
            if world > 1:   # a rank that failed alone cannot rejoin the others' collectives: stop the secondaries here
                if rank == 0:
                    secondary[name] = r2
                break
        if rank == 0:
            if "error" not in r2:
                w2 = WORKLOADS[name]
                r2 = dict(config=config_of(name, w2, args.gpus, r2["iters"], r2["levels"]), value=r2["value"], unit="DOF/s",
                          ms_per_step=r2["ms_per_step"], vcycle_ms=r2["vcycle_ms"], e2e=r2["e2e"], roofline=r2["roofline"],
                          kernels=r2["kernels"], cpu_baseline=r2["cpu_baseline"], parity=r2["parity"],
                          true_residual_rel=r2["true_residual_rel"], host_setup_s=r2["host_setup_s"], gpu_launches=r2["gpu_launches"],
                          **({"krylov": r2["krylov"]} if "krylov" in r2 else {}))
            secondary[name] = r2

    if rank == 0:
        parity = dict(rec["parity"], small=small)
        line = dict(
            metric="amg_pcg_solve_dof_per_s", value=rec["value"], unit="DOF/s", n_gpus=args.gpus,
            steps=args.steps, warmup=args.warmup, ms_per_step=rec["ms_per_step"], higher_is_better=True, scaling="strong",
            vs_baseline=None, dtype="f64", data="synthetic",
            config=config_of(args.workload, wl, args.gpus, rec["iters"], rec["levels"]),
            notes=dict(l2="working set >> 126 MB L2 (no flush needed between solves; kernel timings flush L2 before every launch)",
                       timing="CUDA events inside libpamg around each solve, summed over steps, max over ranks",
                       host_setup_s=rec["host_setup_s"], host_setup=rec["host_setup"]),
            vcycle_ms=rec["vcycle_ms"], wall_ms_per_step=rec["wall_ms_per_step"], true_residual_rel=rec["true_residual_rel"],
            solution_max_err=rec["solution_max_err"], roofline=rec["roofline"], kernels=rec["kernels"], e2e=rec["e2e"],
            gpu_launches=rec["gpu_launches"], clocks=rec["clocks"], cpu_baseline=rec["cpu_baseline"], parity=parity,
            secondary=secondary)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
