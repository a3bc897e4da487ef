"""Per-kernel HBM throughput of every SpMV family on the device-resident hierarchy (1 GPU).
  python scripts/kernel_sweep.py [n=256] [out.json]
Algorithmic bytes follow DESIGN.md / SURVEY.md 8d (fp64 values, int32 columns + row pointers,
each vector element once).  L2 is flushed before every timed launch."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from parallel_amg_b200 import _lib as L  # noqa: E402

n1 = int(sys.argv[1]) if len(sys.argv) > 1 else 256
out = sys.argv[2] if len(sys.argv) > 2 else None
PEAK = 6548.2
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass

c = L.Context(1)
t0 = time.time()
c.gallery_poisson((n1, n1, n1), (1, 1, 1))
c.setup()
print(f"setup {time.time() - t0:.1f}s levels={c.num_levels()}", flush=True)
n, nnz = c.global_size()
rng = np.random.default_rng(1)
b = c.host_matvec_global(rng.uniform(-1, 1, n))

CONFIGS = {
    "auto": dict(spmv_format=L.FORMAT_AUTO),
    "csr": dict(spmv_format=L.FORMAT_CSR),
    "stream": dict(spmv_format=L.FORMAT_STREAM),
    "sell1": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=1, sell_sigma=1),
    "sell2": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=2, sell_sigma=1),
    "sell1-auto": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=1, sell_sigma=0),
    "sell2-auto": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=2, sell_sigma=0),
}
# A/B switches of the engine (read at device_init): name -> environment
ENVS = {
    "auto-novi": dict(PAMG_VALUE_INDEX="0"),       # fp64 values everywhere (round-2 kernels)
    "auto-vi8only": dict(PAMG_VALUE_INDEX="1"),    # one-byte indices only (no wide dictionaries on the coarse levels)
}
for k in ENVS:
    CONFIGS[k] = dict(spmv_format=L.FORMAT_AUTO)
if len(sys.argv) > 3:
    CONFIGS = {k: v for k, v in CONFIGS.items() if k in sys.argv[3].split(",")}
else:
    CONFIGS = {k: v for k, v in CONFIGS.items() if k not in ENVS}
res = {}
for name, kw in CONFIGS.items():
    os.environ.pop("PAMG_VALUE_INDEX", None)
    os.environ.update(ENVS.get(name, {}))
    c.set_kernel_options(**kw)
    c.device_init()
    c.load_rhs([b])
    for _ in range(2):
        it, hist, ok = c.pcg_resident(1e-8, 200, True)
    st = c.stats()
    row = dict(iters=it, solve_ms=st.solve_ms, vcycle_ms=float(np.mean(c.time_kernel(5, 0, 13, False)[3:])))
    for lvl in range(min(int(os.environ.get('SWEEP_LEVELS', '2')), c.num_levels() - 1)):
        info = c.level_info(lvl, 0)
        nr, nc = info.n_own, info.n_own_coarse
        a_b = 12 * info.nnz[0] + 4 * (nr + 1) + 16 * nr
        p_b = 12 * info.nnz[2] + 4 * (nr + 1) + 8 * nc + 16 * nr
        r_b = 12 * info.nnz[4] + 4 * (nc + 1) + 8 * nr + 8 * nc
        algo = {0: ("spmv", a_b), 1: ("jacobi", a_b + 16 * nr), 2: ("resid+restrict", a_b + 8 * nr + r_b), 3: ("prolong", p_b)}
        if lvl == 0:
            algo.update({6: ("spmv+dot", a_b), 7: ("jacobi+dot", a_b + 16 * nr)})
        for kind, (kn, nb) in algo.items():
            ms = float(np.mean(c.time_kernel(kind, lvl, 9, True)[2:]))
            row[f"L{lvl}.{kn}"] = dict(ms=round(ms, 4), gbs=round(nb / ms / 1e6, 1), frac=round(nb / ms / 1e6 / PEAK, 3))
    try:
        ref_ms = float(np.mean(c.time_kernel(8, 0, 9, True)[2:]))
        row["stream_ref"] = dict(ms=round(ref_ms, 4), gbs=round(2 * (256 << 20) / ref_ms / 1e6, 1))
    except Exception:
        pass
    row["fill"] = [round(st.sell_fill[l], 3) for l in range(c.num_levels())]
    row["value_indexed"] = [int(st.value_indexed[l]) for l in range(c.num_levels())]
    res[name] = row
    print(name, json.dumps(row), flush=True)
if out:
    json.dump(res, open(out, "w"), indent=1)
