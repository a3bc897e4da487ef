"""torchrun worker: one rank per GPU, peer-memory halos.  Parity of SpMV / V-cycle / PCG against the
oracle (each rank rebuilds the small oracle problem itself).  Prints MP_GPU_OK on success."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import amg_oracle as O
    from parallel_amg_b200 import _lib as L
    from parallel_amg_b200.distributed import connect_parts
    from util import det_vector, product_options
    pp = {2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}[world]
    # (dims, oracle options, kernel options, environment switches of the engine)
    cases = (((24, 20, 16), {}, {}, {}), ((40, 40, 40), {}, {}, {}), ((24, 20, 16), {"smoother": "chebyshev", "cheb_degree": 2}, {}, {}),
             ((40, 40, 40), {}, dict(spmv_format=L.FORMAT_SELL), {}), ((24, 20, 16), {}, dict(spmv_format=L.FORMAT_CSR), {}),
             ((40, 40, 40), {"smoother": "l1jacobi"}, dict(spmv_format=L.FORMAT_SELL, sell_sigma=128, sell_rows_per_thread=1), {}),
             ((24, 20, 16), {}, dict(fuse_halo=0), {}),
             # SELL with distributed coarse levels (two sweeps, Chebyshev degree 3, defaults); l1-Jacobi and sigma 256 with no replicated tail
             ((40, 40, 40), {"nu_pre": 2, "nu_post": 2}, dict(spmv_format=L.FORMAT_SELL, tail_rows=600), {}),
             ((40, 40, 40), {"smoother": "chebyshev", "cheb_degree": 3}, dict(spmv_format=L.FORMAT_SELL, tail_rows=600), {}),
             ((40, 40, 40), {}, dict(spmv_format=L.FORMAT_SELL, tail_rows=600), {}),
             ((48, 40, 36), {"smoother": "l1jacobi"}, dict(spmv_format=L.FORMAT_SELL, tail_rows=0), {}),
             ((48, 40, 36), {}, dict(spmv_format=L.FORMAT_SELL, sell_sigma=256, tail_rows=0), {}),
             # separate convergence check / W-cycle with a replicated tail / no pre-smoothing
             ((40, 40, 40), {}, {}, {"PAMG_FOLD_CHECK": "0"}),
             ((40, 40, 40), {"cycle": "w", "coarse_size": 40}, dict(tail_rows=600), {}),
             ((40, 40, 40), {"nu_pre": 0, "nu_post": 2}, {}, {}))
    switches = ("PAMG_FOLD_CHECK",)
    for dims, oopts, kopts, env in cases:
        for k in switches:
            os.environ.pop(k, None)
        os.environ.update(env)
        A = O.poisson_fd(dims)
        owner = O.uniform_partition(pp, dims)
        h = O.build(A, owner, world, oopts)
        c = L.Context(world)
        c.gallery_poisson(dims, pp)
        c.setup(product_options(c, oopts, **kopts))
        connect_parts(c, rank, world, local)
        assert c.stats().fused_halo == kopts.get("fuse_halo", 1)
        n = A.shape[0]
        lev = h["levels"][0]
        mine = lev["parts"][rank]["own_to_global"]

        def parts(v):
            return [v[mine] if p == rank else None for p in range(world)]

        for l, levl in enumerate(h["levels"]):
            ng = h["global"]["levels"][l]["A"].shape[0]
            x = det_vector(ng, 5 + l)
            own_l = levl["parts"][rank]["own_to_global"]
            y = c.spmv(l, [x[own_l] if p == rank else None for p in range(world)])[rank]
            ref = (h["global"]["levels"][l]["A"] @ x)[own_l]
            assert np.abs(y - ref).max() <= 1e-12 * np.abs(ref).max(), ("spmv", l)
        b = det_vector(n, 9)
        z = c.vcycle(parts(b))[rank]
        z_ref = O.vcycle(h, O.pvector_from_global(lev, b))[rank][:len(mine)]
        zn = max(np.abs(r).max() for r in O.vcycle(h, O.pvector_from_global(lev, b)))
        assert np.abs(z - z_ref).max() <= 1e-12 * zn, ("vcycle", np.abs(z - z_ref).max())
        rhs = A @ det_vector(n, 1)
        xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, rhs))
        for rep in range(3):  # repeated solves exercise the epoch / parity protocol across solves
            x, it, hist, ok = c.pcg(parts(rhs))
            assert ok and it == it_ref, (it, it_ref)
            assert np.allclose(hist, hist_ref, rtol=1e-7)
            assert np.abs(x[rank] - xs[rank][:len(mine)]).max() <= 1e-9
        d = c.dot(0, parts(b), parts(rhs))
        assert abs(d - float(b @ rhs)) <= 1e-12 * np.abs(b * rhs).sum()
        loc = [np.concatenate([b[mine], np.full(len(lev["parts"][rank]["ghost_to_global"]), np.nan)]) if p == rank else None
               for p in range(world)]
        c.consistent(0, loc)
        assert np.array_equal(loc[rank][len(mine):], b[lev["parts"][rank]["ghost_to_global"]])
        dist.barrier()
        c.close()
        if rank == 0:
            print("case ok", dims, oopts, {k: v for k, v in kopts.items()}, env, flush=True)
    if rank == 0:
        print("MP_GPU_OK", world, flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
