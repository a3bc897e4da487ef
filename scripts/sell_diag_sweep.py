"""Level-0 kernel times of the headline workload (3-D Poisson, one part, AUTO formats) with the L2 flushed before every launch,
the bytes the storage format of A0 has to move per launch, and the resulting fraction of the HBM rate.

    python scripts/sell_diag_sweep.py [--tree DIR] [--n 256] [--reps 25]

--tree DIR imports parallel_amg_b200 from another checkout (with its own built libpamg.so), so that two builds can be timed in
one session.  Bytes per launch, n = rows, nd = stored diagonals of the implied-column layout (else 5 B per entry of the
value-indexed layout: int32 column + index byte):
    spmv (kind 0) and spmv + fused p.q (kind 6):           matrix + 16 n   (x read, y written)
    jacobi sweep (kind 1) and sweep + fused r.z (kind 7):  matrix + 32 n   (x, b, w read, x_new written)
    residual + restriction (kind 2):                       matrix + 24 n   (x, b read, r written)
                                                           + 5 nnz(R) + 8 n + 24 n_coarse  (R pass: r read, w_c read, b_c and x_c written)
The fraction is taken against MEASURED_PEAKS.json hbm_gbs when the file exists, and always against the reference stream
(kind 8: read + write of a 256 MiB buffer) timed in the same run."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=None, help="checkout whose parallel_amg_b200 (and libpamg.so) to time")
    ap.add_argument("--n", type=int, default=256, help="nodes per direction")
    ap.add_argument("--reps", type=int, default=25, help="launches per kernel (the first three are dropped)")
    args = ap.parse_args()
    tree = os.path.abspath(args.tree or ROOT)
    sys.path.insert(0, tree)
    from parallel_amg_b200 import _lib as L

    n = args.n
    c = L.Context(1)
    c.gallery_poisson((n, n, n), (1, 1, 1))
    c.setup(c.default_options())
    c.device_init()
    st = c.stats()
    info = c.level_info(0, 0)
    rows, nnz, nc, nnz_r = info.n_own, info.nnz[L.A_OO], info.n_own_coarse, info.nnz[L.R_OO]
    diag = bool(st.value_indexed[0] & 64)
    if diag:
        nd = len(c.layout_sell_diag(0, 0)["off"])
        matrix, fmt = nd * rows, f"implied columns, {nd} diagonals x 1 B"
    elif st.value_indexed[0] & 1:
        matrix, fmt = 5 * nnz, "value-indexed SELL, int32 column + 1 B"
    else:
        matrix, fmt = 12 * nnz, "fp64 values + int32 columns"
    r_matrix = (5 if st.value_indexed[0] & 4 else 12) * nnz_r
    kinds = {0: ("spmv", matrix + 16 * rows), 6: ("spmv + p.q", matrix + 16 * rows), 1: ("jacobi sweep", matrix + 32 * rows),
             7: ("jacobi sweep + r.z", matrix + 32 * rows), 2: ("residual + restriction", matrix + 24 * rows + r_matrix + 8 * rows + 24 * nc)}

    stream_ms = float(np.median(c.time_kernel(8, 0, args.reps, True)[3:]))
    stream_gbs = 2 * (256 << 20) / (stream_ms * 1e-3) / 1e9
    peak = None
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peak = float(json.load(fh)["hbm_gbs"])
    except (OSError, KeyError, ValueError):
        pass
    head = dict(tree=tree, n=rows, nnz=int(nnz), format=fmt, value_indexed=int(st.value_indexed[0]), stream_gbs=round(stream_gbs, 1),
                measured_peak_gbs=peak)
    print(json.dumps(head))
    print(f"{'kernel':24s} {'ms (median)':>11s} {'ms (min)':>9s} {'GB moved':>9s} {'GB/s':>7s} {'of stream':>9s} {'of peak':>8s}")
    for kind, (name, nbytes) in kinds.items():
        ms = c.time_kernel(kind, 0, args.reps, True)[3:]
        med = float(np.median(ms))
        gbs = nbytes / (med * 1e-3) / 1e9
        rec = dict(kernel=name, kind=kind, ms_median=round(med, 4), ms_min=round(float(np.min(ms)), 4), bytes=int(nbytes),
                   gbs=round(gbs, 1), frac_stream=round(gbs / stream_gbs, 3), frac_peak=round(gbs / peak, 3) if peak else None)
        print(f"{name:24s} {med:11.4f} {float(np.min(ms)):9.4f} {nbytes / 1e9:9.3f} {gbs:7.0f} {rec['frac_stream']:9.3f} "
              f"{rec['frac_peak'] if peak else '-':>8}")
        print(json.dumps(rec))
    c.close()


if __name__ == "__main__":
    main()
