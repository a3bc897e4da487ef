"""ctypes binding of libpamg.so (include/pamg.h).  The library is built in-tree by
parallel_amg_b200/build.py; if it is missing this module raises — there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpamg.so")

OK, ERR_ARG, ERR_CUDA, ERR_NOGPU, ERR_COMM, ERR_NOTCONV, ERR_ALLOC = 0, -1, -2, -3, -4, -5, -6
SMOOTHER_JACOBI, SMOOTHER_L1JACOBI, SMOOTHER_CHEBYSHEV = 0, 1, 2
FORMAT_AUTO, FORMAT_CSR, FORMAT_STREAM, FORMAT_SELL, FORMAT_SELL_DIAG = 0, 1, 2, 3, 4
CYCLE_V, CYCLE_W = 0, 1
A_OO, A_OG, P_OO, P_OG, R_OO, R_OG = range(6)
BLOCK_NAMES = ("A_oo", "A_og", "P_oo", "P_og", "R_oo", "R_og")


class PamgError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"pamg status {status}: {msg}")
        self.status = status


class Options(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("eps_strength", C.c_double), ("coarse_size", C.c_int32),
        ("max_levels", C.c_int32), ("smoother", C.c_int32), ("omega_jacobi", C.c_double),
        ("nu_pre", C.c_int32), ("nu_post", C.c_int32), ("cheb_degree", C.c_int32),
        ("cheb_lo_frac", C.c_double), ("cheb_hi_frac", C.c_double), ("spmv_format", C.c_int32),
        ("use_graph", C.c_int32), ("lanes_per_row", C.c_int32), ("tail_rows", C.c_int32), ("sell_sigma", C.c_int32), ("sell_rows_per_thread", C.c_int32), ("fuse_halo", C.c_int32),
        ("cycle", C.c_int32),
    ]


class LevelInfo(C.Structure):
    _fields_ = [
        ("n_global", C.c_int64), ("n_own", C.c_int64), ("n_ghost", C.c_int64), ("n_own_coarse", C.c_int64),
        ("nnz", C.c_int64 * 6), ("n_recv_nbrs", C.c_int32), ("n_send_nbrs", C.c_int32), ("n_send", C.c_int64),
        ("rho", C.c_double), ("omega_p", C.c_double),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("iters", C.c_int32), ("converged", C.c_int32), ("r0_norm", C.c_double), ("r_norm", C.c_double),
        ("solve_ms", C.c_double), ("vcycle_ms", C.c_double), ("kernel_launches", C.c_int64),
        ("n_levels", C.c_int32), ("format", C.c_int32 * 16), ("lanes", C.c_int32 * 16),
        ("format_p", C.c_int32 * 16), ("format_r", C.c_int32 * 16), ("sell_fill", C.c_double * 16), ("fused_halo", C.c_int32), ("tail_level", C.c_int32),
        ("value_indexed", C.c_int32 * 16),
    ]


_P = C.POINTER
_i64p, _i32p, _f64p = _P(C.c_int64), _P(C.c_int32), _P(C.c_double)
_vecs = _P(_f64p)
_ctx = C.c_void_p

# name -> argtypes (restype is int unless listed in _RESTYPE); also the list tests check exports against
PROTOTYPES = {
    "pamg_default_options": [_P(Options)],
    "pamg_create": [C.c_int32, _P(_ctx)],
    "pamg_destroy": [_ctx],
    "pamg_last_error": [_ctx],
    "pamg_set_part_rows": [_ctx, C.c_int32, C.c_int64, _i64p, _i64p, _i64p, _f64p],
    "pamg_set_matrix_global": [_ctx, C.c_int64, _i64p, _i64p, _f64p, _i32p],
    "pamg_gallery_poisson": [_ctx, C.c_int32, _i64p, _i32p],
    "pamg_gallery_diffusion_jump": [_ctx, C.c_int32, _i64p, _i32p, C.c_int32, C.c_double, C.c_double],
    "pamg_gallery_elasticity": [_ctx, _i64p, _i32p, C.c_double, C.c_double],
    "pamg_set_near_nullspace": [_ctx, C.c_int32, C.c_int32, _f64p],
    "pamg_get_near_nullspace": [_ctx, _i32p, _i32p, _f64p],
    "pamg_uniform_partition": [C.c_int32, _i64p, _i32p, _i32p],
    "pamg_host_matvec_global": [_ctx, _f64p, _f64p],
    "pamg_global_size": [_ctx, _i64p, _i64p],
    "pamg_set_num_threads": [C.c_int32],
    "pamg_setup": [_ctx, _P(Options)],
    "pamg_hierarchy_begin": [_ctx, C.c_int32, _P(Options)],
    "pamg_level_upload": [_ctx, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _i64p, _i64p, _i32p, C.c_int64, C.c_int64,
                          _P(_i64p), _P(_i32p), _P(_f64p), C.c_double],
    "pamg_coarse_upload": [_ctx, C.c_int64, _f64p],
    "pamg_hierarchy_end": [_ctx],
    "pamg_layout_sell": [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i64p, _i64p, _i32p, _i32p, _i32p, _f64p, _i32p],
    "pamg_layout_sell_values": [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i32p, _i64p, _f64p, _P(C.c_uint8)],
    "pamg_layout_sell_diag": [_ctx, C.c_int32, C.c_int32, C.c_int32, _i32p, _i32p, _i64p, _f64p, _P(C.c_uint8)],
    "pamg_layout_stream": [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i64p, _i32p, _i32p],
    "pamg_layout_boundary": [_ctx, C.c_int32, C.c_int32, C.c_int32, _i64p, _i64p, _i32p, _i32p, _i32p, _i32p, _i32p, _f64p,
                             _P(C.c_uint8)],
    "pamg_hierarchy_save": [_ctx, C.c_char_p],
    "pamg_hierarchy_load": [_ctx, C.c_char_p, C.c_int32],
    "pamg_num_levels": [_ctx, _i32p],
    "pamg_get_level_info": [_ctx, C.c_int32, C.c_int32, _P(LevelInfo)],
    "pamg_get_index_maps": [_ctx, C.c_int32, C.c_int32, _i64p, _i64p, _i32p],
    "pamg_get_block": [_ctx, C.c_int32, C.c_int32, C.c_int32, _i64p, _i32p, _f64p],
    "pamg_get_aggregates": [_ctx, C.c_int32, C.c_int32, _i32p],
    "pamg_get_halo_plan": [_ctx, C.c_int32, C.c_int32, _i32p, _i32p, _i32p, _i32p, _i32p, _i32p, _i32p],
    "pamg_get_coarse_inverse": [_ctx, _i64p, _f64p],
    "pamg_get_diag": [_ctx, C.c_int32, C.c_int32, _f64p, _f64p],
    "pamg_set_kernel_options": [_ctx, _P(Options)],
    "pamg_device_init": [_ctx, C.c_int32, _i32p, _i32p],
    "pamg_comm_handle_bytes": [],
    "pamg_comm_export": [_ctx, C.c_int32, C.c_void_p],
    "pamg_comm_import": [_ctx, C.c_int32, C.c_void_p],
    "pamg_comm_connect": [_ctx],
    "pamg_spmv": [_ctx, C.c_int32, _vecs, _vecs],
    "pamg_consistent": [_ctx, C.c_int32, _vecs],
    "pamg_assemble": [_ctx, C.c_int32, _vecs],
    "pamg_smooth": [_ctx, C.c_int32, C.c_int32, _vecs, _vecs],
    "pamg_residual_restrict": [_ctx, C.c_int32, _vecs, _vecs, _vecs, _vecs],
    "pamg_prolong_correct": [_ctx, C.c_int32, _vecs, _vecs],
    "pamg_dot": [_ctx, C.c_int32, _vecs, _vecs, _f64p],
    "pamg_vcycle": [_ctx, _vecs, _vecs],
    "pamg_pcg": [_ctx, _vecs, _vecs, C.c_double, C.c_int32, C.c_int32, _i32p, _f64p],
    "pamg_fcg": [_ctx, _vecs, _vecs, C.c_double, C.c_int32, _i32p, _f64p],
    "pamg_fgmres": [_ctx, _vecs, _vecs, C.c_double, C.c_int32, C.c_int32, C.c_int32, _i32p, _f64p],
    "pamg_load_rhs": [_ctx, _vecs],
    "pamg_pcg_resident": [_ctx, C.c_double, C.c_int32, C.c_int32, _i32p, _f64p],
    "pamg_read_solution": [_ctx, _vecs],
    "pamg_time_kernel": [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P(C.c_float)],
    "pamg_get_stats": [_ctx, _P(Stats)],
    "pamg_trace_enable": [_ctx, C.c_int32],
    "pamg_trace_read": [_ctx, C.c_int32, _P(C.c_uint64), C.c_int32, _i32p],
    "pamg_trace_names": [_ctx, C.c_char_p, C.c_int32],
    "pamg_set_rhs_capacity": [_ctx, C.c_int32],
    "pamg_spmv_multi": [_ctx, C.c_int32, C.c_int32, _vecs, _vecs],
    "pamg_vcycle_multi": [_ctx, C.c_int32, _vecs, _vecs],
    "pamg_time_kernel_multi": [_ctx, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P(C.c_float)],
    "pamg_pcg_multi": [_ctx, C.c_int32, _vecs, _vecs, C.c_double, C.c_int32, C.c_int32, _i32p, _i32p, _f64p],
}
_RESTYPE = {"pamg_set_num_threads": None, "pamg_default_options": None, "pamg_destroy": None, "pamg_last_error": C.c_char_p,
            "pamg_comm_handle_bytes": C.c_int32}

_lib = None


def load():
    """dlopen libpamg.so and attach prototypes; raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -m parallel_amg_b200.build` "
                          "(the CUDA library is mandatory; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, args in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _RESTYPE.get(name, C.c_int)
    _lib = lib
    return lib


def set_num_threads(n):
    """OpenMP threads of the host-side setup (torchrun exports OMP_NUM_THREADS=1)."""
    load().pamg_set_num_threads(int(n))


def _ptr(a, ctype):
    if a is None:
        return None
    return a.ctypes.data_as(C.POINTER(ctype))


def _as(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


class Context:
    """Thin numpy-facing wrapper of a pamg_ctx*.  One context = one partitioned linear system +
    its AMG hierarchy + (after device_init) its device-resident copy."""

    def __init__(self, nparts):
        self.lib = load()
        self.nparts = int(nparts)
        self._h = _ctx()
        st = self.lib.pamg_create(self.nparts, C.byref(self._h))
        if st != OK:
            raise PamgError(st, "pamg_create failed")
        self._info_cache = {}

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.pamg_destroy(self._h)
            self._h = _ctx()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, st, allow=()):
        if st != OK and st not in allow:
            raise PamgError(st, self.lib.pamg_last_error(self._h).decode(errors="replace"))
        return st

    # ---- options ----
    def default_options(self, **kw):
        o = Options()
        self.lib.pamg_default_options(C.byref(o))
        for k, v in kw.items():
            if not hasattr(o, k):
                raise KeyError(k)
            setattr(o, k, v)
        return o

    # ---- problem ----
    def gallery_poisson(self, nodes_per_dir, parts_per_dir):
        n = _as(nodes_per_dir, np.int64)
        p = _as(parts_per_dir, np.int32)
        self._ck(self.lib.pamg_gallery_poisson(self._h, len(n), _ptr(n, C.c_int64), _ptr(p, C.c_int32)))

    def gallery_diffusion_jump(self, nodes_per_dir, parts_per_dir, blocks=8, kmax=1.0e4, eps_z=1.0e-3):
        n = _as(nodes_per_dir, np.int64)
        p = _as(parts_per_dir, np.int32)
        self._ck(self.lib.pamg_gallery_diffusion_jump(self._h, len(n), _ptr(n, C.c_int64), _ptr(p, C.c_int32),
                                                      int(blocks), float(kmax), float(eps_z)))

    def gallery_elasticity(self, nodes_per_dir, parts_per_dir, E=1.0, nu=0.25):
        n = _as(nodes_per_dir, np.int64)
        p = _as(parts_per_dir, np.int32)
        assert len(n) == 3 and len(p) == 3
        self._ck(self.lib.pamg_gallery_elasticity(self._h, _ptr(n, C.c_int64), _ptr(p, C.c_int32), float(E), float(nu)))

    def set_near_nullspace(self, block_size, B):
        if B is None:
            self._ck(self.lib.pamg_set_near_nullspace(self._h, 1, 0, None))
            return
        B = _as(B, np.float64)
        self._ck(self.lib.pamg_set_near_nullspace(self._h, int(block_size), B.shape[1], _ptr(B, C.c_double)))

    def near_nullspace(self):
        bs, k = C.c_int32(), C.c_int32()
        self._ck(self.lib.pamg_get_near_nullspace(self._h, C.byref(bs), C.byref(k), None))
        n, _ = self.global_size()
        B = np.zeros((n, max(k.value, 0)))
        if k.value > 0:
            self._ck(self.lib.pamg_get_near_nullspace(self._h, C.byref(bs), C.byref(k), _ptr(B, C.c_double)))
        return bs.value, B

    def set_matrix_global(self, indptr, indices, data, owner):
        ip, ix, d, ow = _as(indptr, np.int64), _as(indices, np.int64), _as(data, np.float64), _as(owner, np.int32)
        self._ck(self.lib.pamg_set_matrix_global(self._h, len(ip) - 1, _ptr(ip, C.c_int64), _ptr(ix, C.c_int64),
                                                 _ptr(d, C.c_double), _ptr(ow, C.c_int32)))

    def set_part_rows(self, part, own_to_global, indptr, col_gid, data):
        o, ip, ix, d = _as(own_to_global, np.int64), _as(indptr, np.int64), _as(col_gid, np.int64), _as(data, np.float64)
        self._ck(self.lib.pamg_set_part_rows(self._h, int(part), len(o), _ptr(o, C.c_int64), _ptr(ip, C.c_int64),
                                             _ptr(ix, C.c_int64), _ptr(d, C.c_double)))

    def global_size(self):
        n, nnz = C.c_int64(), C.c_int64()
        self._ck(self.lib.pamg_global_size(self._h, C.byref(n), C.byref(nnz)))
        return n.value, nnz.value

    def host_matvec_global(self, x):
        x = _as(x, np.float64)
        y = np.empty_like(x)
        self._ck(self.lib.pamg_host_matvec_global(self._h, _ptr(x, C.c_double), _ptr(y, C.c_double)))
        return y

    # ---- setup ----
    def setup(self, opts=None):
        self._info_cache.clear()
        self._ck(self.lib.pamg_setup(self._h, C.byref(opts) if opts is not None else None))

    def upload_hierarchy(self, levels, coarse_inv, opts=None, rho=None):
        """levels[l][p] = dict(own_to_global, ghost_to_global, ghost_to_owner, A_oo, A_og[, P_oo, P_og,
        R_oo, R_og]) with scipy CSR blocks (the layout oracle/amg_oracle.py localize() produces)."""
        self._info_cache.clear()
        L = len(levels)
        self._ck(self.lib.pamg_hierarchy_begin(self._h, L, C.byref(opts) if opts is not None else None))
        for l, parts in enumerate(levels):
            for p, d in enumerate(parts):
                own = _as(d["own_to_global"], np.int64)
                gh = _as(d["ghost_to_global"], np.int64)
                gho = _as(d["ghost_to_owner"], np.int32)
                nxt = levels[l + 1][p] if l + 1 < L else None
                noc = len(nxt["own_to_global"]) if nxt else 0
                ngc = len(nxt["ghost_to_global"]) if nxt else 0
                keep = []
                rp = (_i64p * 6)()
                cp = (_i32p * 6)()
                vp = (_f64p * 6)()
                for b, name in enumerate(BLOCK_NAMES):
                    m = d.get(name)
                    if m is None:
                        continue
                    ip, ix, dd = _as(m.indptr, np.int64), _as(m.indices, np.int32), _as(m.data, np.float64)
                    keep += [ip, ix, dd]
                    rp[b], cp[b], vp[b] = _ptr(ip, C.c_int64), _ptr(ix, C.c_int32), _ptr(dd, C.c_double)
                self._ck(self.lib.pamg_level_upload(self._h, l, p, len(own), len(gh), _ptr(own, C.c_int64),
                                                    _ptr(gh, C.c_int64), _ptr(gho, C.c_int32), noc, ngc, rp, cp, vp,
                                                    float(rho[l]) if rho is not None and rho[l] is not None else 0.0))
        inv = _as(coarse_inv, np.float64)
        self._ck(self.lib.pamg_coarse_upload(self._h, inv.shape[0], _ptr(inv, C.c_double)))
        self._ck(self.lib.pamg_hierarchy_end(self._h))

    def hierarchy_save(self, path):
        self._ck(self.lib.pamg_hierarchy_save(self._h, str(path).encode()))

    def hierarchy_load(self, path, keep_part=-1):
        self._info_cache.clear()
        self._ck(self.lib.pamg_hierarchy_load(self._h, str(path).encode(), int(keep_part)))

    # ---- queries ----
    def num_levels(self):
        n = C.c_int32()
        self._ck(self.lib.pamg_num_levels(self._h, C.byref(n)))
        return n.value

    def level_info(self, level, part):
        key = (level, part)
        if key not in self._info_cache:
            info = LevelInfo()
            self._ck(self.lib.pamg_get_level_info(self._h, level, part, C.byref(info)))
            self._info_cache[key] = info
        return self._info_cache[key]

    def index_maps(self, level, part):
        i = self.level_info(level, part)
        own, gh, gho = np.empty(i.n_own, np.int64), np.empty(i.n_ghost, np.int64), np.empty(i.n_ghost, np.int32)
        self._ck(self.lib.pamg_get_index_maps(self._h, level, part, _ptr(own, C.c_int64), _ptr(gh, C.c_int64),
                                              _ptr(gho, C.c_int32)))
        return own, gh, gho

    def block(self, level, part, which):
        """(indptr int64, indices int32, data float64, shape)"""
        i = self.level_info(level, part)
        nr = i.n_own_coarse if which >= R_OO else i.n_own
        nnz = i.nnz[which]
        ip, ix, d = np.zeros(nr + 1, np.int64), np.empty(nnz, np.int32), np.empty(nnz, np.float64)
        self._ck(self.lib.pamg_get_block(self._h, level, part, which, _ptr(ip, C.c_int64), _ptr(ix, C.c_int32),
                                         _ptr(d, C.c_double)))
        return ip, ix, d

    def aggregates(self, level, part):
        i = self.level_info(level, part)
        a = np.empty(i.n_own, np.int32)
        self._ck(self.lib.pamg_get_aggregates(self._h, level, part, _ptr(a, C.c_int32)))
        return a

    def halo_plan(self, level, part):
        i = self.level_info(level, part)
        r = [np.empty(i.n_recv_nbrs, np.int32) for _ in range(3)]
        s = [np.empty(i.n_send_nbrs, np.int32) for _ in range(3)]
        idx = np.empty(i.n_send, np.int32)
        self._ck(self.lib.pamg_get_halo_plan(self._h, level, part, *[_ptr(a, C.c_int32) for a in r],
                                             *[_ptr(a, C.c_int32) for a in s], _ptr(idx, C.c_int32)))
        return dict(recv_part=r[0], recv_slot0=r[1], recv_count=r[2], send_part=s[0], send_slot0=s[1],
                    send_count=s[2], send_idx=idx)

    def coarse_inverse(self):
        n = C.c_int64()
        self._ck(self.lib.pamg_get_coarse_inverse(self._h, C.byref(n), None))
        inv = np.empty((n.value, n.value), np.float64)
        self._ck(self.lib.pamg_get_coarse_inverse(self._h, C.byref(n), _ptr(inv, C.c_double)))
        return inv

    def diag(self, level, part):
        i = self.level_info(level, part)
        d, d1 = np.empty(i.n_own), np.empty(i.n_own)
        self._ck(self.lib.pamg_get_diag(self._h, level, part, _ptr(d, C.c_double), _ptr(d1, C.c_double)))
        return d, d1

    # ---- device layouts (host-side conversions, no GPU needed) ----
    def layout_sell(self, level, part, which, rows_per_slice=64, sigma=1):
        ns, st, pm = C.c_int64(), C.c_int64(), C.c_int32()
        self._ck(self.lib.pamg_layout_sell(self._h, level, part, which, rows_per_slice, sigma, C.byref(ns), C.byref(st),
                                           C.byref(pm), None, None, None, None))
        i = self.level_info(level, part)
        nr = i.n_own_coarse if which >= R_OO else i.n_own
        off, col, val = np.zeros(ns.value + 1, np.int32), np.zeros(st.value, np.int32), np.zeros(st.value)
        perm = np.zeros(nr, np.int32)
        self._ck(self.lib.pamg_layout_sell(self._h, level, part, which, rows_per_slice, sigma, C.byref(ns), C.byref(st),
                                           C.byref(pm), _ptr(off, C.c_int32), _ptr(col, C.c_int32), _ptr(val, C.c_double),
                                           _ptr(perm, C.c_int32)))
        return dict(slice_off=off, col=col, val=val, perm=perm, permuted=bool(pm.value), C=rows_per_slice)

    def layout_sell_values(self, level, part, which, rows_per_slice=64, sigma=1):
        """(dict[4096], vidx[stored] as uint8 or uint16) of the value-indexed SELL storage, or None when the block has more than 4095
        distinct values; vidx.dtype tells the index width."""
        ix, st = C.c_int32(), C.c_int64()
        self._ck(self.lib.pamg_layout_sell_values(self._h, level, part, which, rows_per_slice, sigma, C.byref(ix), C.byref(st), None, None))
        if not ix.value:
            return None
        d, v = np.zeros(4096), np.zeros(st.value * ix.value, np.uint8)
        self._ck(self.lib.pamg_layout_sell_values(self._h, level, part, which, rows_per_slice, sigma, C.byref(ix), C.byref(st),
                                                  _ptr(d, C.c_double), _ptr(v, C.c_uint8)))
        return d, (v if ix.value == 1 else v.view("<u2"))

    def layout_sell_diag(self, level, part, which=A_OO):
        """SELL with implied columns: dict(off, dict[256], idx[stored] uint8; 255 = no entry), or None when the block does not qualify."""
        nd, st = C.c_int32(), C.c_int64()
        self._ck(self.lib.pamg_layout_sell_diag(self._h, level, part, which, C.byref(nd), None, C.byref(st), None, None))
        if not nd.value:
            return None
        off, d, idx = np.zeros(nd.value, np.int32), np.zeros(256), np.zeros(st.value, np.uint8)
        self._ck(self.lib.pamg_layout_sell_diag(self._h, level, part, which, C.byref(nd), _ptr(off, C.c_int32), C.byref(st),
                                                _ptr(d, C.c_double), _ptr(idx, C.c_uint8)))
        return dict(off=off, dict=d, idx=idx)

    def layout_stream(self, level, part, which, max_rows=1024, max_entries=3069):
        nb = C.c_int64()
        self._ck(self.lib.pamg_layout_stream(self._h, level, part, which, max_rows, max_entries, C.byref(nb), None, None))
        if nb.value < 0:
            return None
        r, e = np.zeros(nb.value + 1, np.int32), np.zeros(nb.value + 1, np.int32)
        self._ck(self.lib.pamg_layout_stream(self._h, level, part, which, max_rows, max_entries, C.byref(nb),
                                             _ptr(r, C.c_int32), _ptr(e, C.c_int32)))
        return r, e

    def layout_boundary(self, level, part, which):
        n, ne, ln = C.c_int64(), C.c_int64(), C.c_int32()
        self._ck(self.lib.pamg_layout_boundary(self._h, level, part, which, C.byref(n), C.byref(ne), C.byref(ln),
                                               None, None, None, None, None, None))
        i = self.level_info(level, part)
        nr = i.n_own_coarse if which >= R_OO else i.n_own
        rows, ptr, mid = np.zeros(n.value, np.int32), np.zeros(n.value + 1, np.int32), np.zeros(n.value, np.int32)
        col, val, skip = np.zeros(ne.value, np.int32), np.zeros(ne.value), np.zeros(max(nr, 1), np.uint8)
        self._ck(self.lib.pamg_layout_boundary(self._h, level, part, which, C.byref(n), C.byref(ne), C.byref(ln),
                                               _ptr(rows, C.c_int32), _ptr(ptr, C.c_int32), _ptr(mid, C.c_int32),
                                               _ptr(col, C.c_int32), _ptr(val, C.c_double), _ptr(skip, C.c_uint8)))
        return dict(rows=rows, ptr=ptr, mid=mid, col=col, val=val, skip=skip[:nr], lanes=ln.value)

    # ---- device ----
    def device_init(self, local_parts=None, device_ids=None):
        lp = _as(range(self.nparts) if local_parts is None else local_parts, np.int32)
        dv = _as([0] * len(lp) if device_ids is None else device_ids, np.int32)
        self.local_parts = [int(p) for p in lp]
        self._ck(self.lib.pamg_device_init(self._h, len(lp), _ptr(lp, C.c_int32), _ptr(dv, C.c_int32)))

    def set_kernel_options(self, **kw):
        """Change spmv_format / lanes_per_row / use_graph / sell_* for the next device_init."""
        o = self.default_options(**kw)
        self._ck(self.lib.pamg_set_kernel_options(self._h, C.byref(o)))

    def comm_export(self, part):
        buf = C.create_string_buffer(self.lib.pamg_comm_handle_bytes())
        self._ck(self.lib.pamg_comm_export(self._h, int(part), buf))
        return buf.raw

    def comm_import(self, part, blob):
        buf = C.create_string_buffer(bytes(blob), len(blob))
        self._ck(self.lib.pamg_comm_import(self._h, int(part), buf))

    def comm_connect(self):
        self._ck(self.lib.pamg_comm_connect(self._h))

    def _vecs(self, arrs, level=None, local=False, writable=False):
        """list (len nparts, None allowed for remote parts) -> double** ; returns (ptr array, keepalive)"""
        out = (_f64p * self.nparts)()
        keep = []
        for p in range(self.nparts):
            a = arrs[p] if arrs is not None else None
            if a is None:
                out[p] = None
                continue
            if writable:
                assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
            else:
                a = _as(a, np.float64)
            keep.append(a)
            out[p] = _ptr(a, C.c_double)
        return out, keep

    def _vecs_multi(self, cols, writable=False):
        """k columns, each a per-part list as pcg() takes -> double*[k * nparts], column j of part p at [j * nparts + p]"""
        out = (_f64p * (len(cols) * self.nparts))()
        keep = []
        for j, col in enumerate(cols):
            ptrs, k = self._vecs(col, writable=writable)
            keep.append((ptrs, k))
            for p in range(self.nparts):
                out[j * self.nparts + p] = ptrs[p]
        return out, keep

    def _new_own(self, level):
        return [np.zeros(self.level_info(level, p).n_own) if p in self.local_parts else None
                for p in range(self.nparts)]

    def spmv(self, level, x):
        y = self._new_own(level)
        xp, k1 = self._vecs(x)
        yp, k2 = self._vecs(y, writable=True)
        self._ck(self.lib.pamg_spmv(self._h, level, xp, yp))
        return y

    def consistent(self, level, v):
        vp, k = self._vecs(v, writable=True)
        self._ck(self.lib.pamg_consistent(self._h, level, vp))
        return v

    def assemble(self, level, v):
        vp, k = self._vecs(v, writable=True)
        self._ck(self.lib.pamg_assemble(self._h, level, vp))
        return v

    def smooth(self, level, nu, b, x):
        x = [None if a is None else np.array(a, dtype=np.float64) for a in x]
        bp, k1 = self._vecs(b)
        xp, k2 = self._vecs(x, writable=True)
        self._ck(self.lib.pamg_smooth(self._h, level, nu, bp, xp))
        return x

    def residual_restrict(self, level, b, x, want_r=True):
        r = self._new_own(level) if want_r else None
        bc = self._new_own(level + 1)
        bp, k1 = self._vecs(b)
        xp, k2 = self._vecs(x)
        rp, k3 = self._vecs(r, writable=True) if want_r else (None, None)
        cp, k4 = self._vecs(bc, writable=True)
        self._ck(self.lib.pamg_residual_restrict(self._h, level, bp, xp, rp, cp))
        return r, bc

    def prolong_correct(self, level, ec, x):
        x = [None if a is None else np.array(a, dtype=np.float64) for a in x]
        ep, k1 = self._vecs(ec)
        xp, k2 = self._vecs(x, writable=True)
        self._ck(self.lib.pamg_prolong_correct(self._h, level, ep, xp))
        return x

    def dot(self, level, u, v):
        up, k1 = self._vecs(u)
        vp, k2 = self._vecs(v)
        out = C.c_double()
        self._ck(self.lib.pamg_dot(self._h, level, up, vp, C.byref(out)))
        return out.value

    def vcycle(self, b):
        x = self._new_own(0)
        bp, k1 = self._vecs(b)
        xp, k2 = self._vecs(x, writable=True)
        self._ck(self.lib.pamg_vcycle(self._h, bp, xp))
        return x

    def pcg(self, b, rtol=1e-8, maxiter=200, precond=True, out=None):
        """out: optional list of preallocated (e.g. pinned) float64 arrays receiving the own values of x."""
        x = out if out is not None else self._new_own(0)
        bp, k1 = self._vecs(b)
        xp, k2 = self._vecs(x, writable=True)
        it = C.c_int32()
        hist = np.zeros(maxiter + 2)
        st = self._ck(self.lib.pamg_pcg(self._h, bp, xp, float(rtol), int(maxiter), int(bool(precond)), C.byref(it),
                                        _ptr(hist, C.c_double)), allow=(ERR_NOTCONV,))
        return x, it.value, hist[:it.value + 1].copy(), st == OK

    def fcg(self, b, rtol=1e-8, maxiter=200, out=None):
        """flexible AMG-preconditioned CG; same results tuple as pcg()."""
        x = out if out is not None else self._new_own(0)
        bp, k1 = self._vecs(b)
        xp, k2 = self._vecs(x, writable=True)
        it = C.c_int32()
        hist = np.zeros(maxiter + 2)
        st = self._ck(self.lib.pamg_fcg(self._h, bp, xp, float(rtol), int(maxiter), C.byref(it), _ptr(hist, C.c_double)),
                      allow=(ERR_NOTCONV,))
        return x, it.value, hist[:it.value + 1].copy(), st == OK

    def fgmres(self, b, rtol=1e-8, maxiter=200, restart=30, precond=True, out=None):
        """restarted flexible GMRES right-preconditioned by one cycle; same results tuple as pcg() (hist = residual estimates)."""
        x = out if out is not None else self._new_own(0)
        bp, k1 = self._vecs(b)
        xp, k2 = self._vecs(x, writable=True)
        it = C.c_int32()
        hist = np.zeros(maxiter + 2)
        st = self._ck(self.lib.pamg_fgmres(self._h, bp, xp, float(rtol), int(maxiter), int(restart), int(bool(precond)),
                                           C.byref(it), _ptr(hist, C.c_double)), allow=(ERR_NOTCONV,))
        return x, it.value, hist[:it.value + 1].copy(), st == OK

    # ---- several right-hand sides (k solve! calls sharing one setup) ----
    def set_rhs_capacity(self, kmax):
        """columns of device state the next device_init allocates (1..8)"""
        self._ck(self.lib.pamg_set_rhs_capacity(self._h, int(kmax)))

    def spmv_multi(self, level, X):
        """X: list of k columns, each a per-part list as spmv() takes; returns the k results (column j == spmv(level, X[j]))"""
        Y = [self._new_own(level) for _ in X]
        xp, k1 = self._vecs_multi(X)
        yp, k2 = self._vecs_multi(Y, writable=True)
        self._ck(self.lib.pamg_spmv_multi(self._h, int(level), len(X), xp, yp))
        return Y

    def vcycle_multi(self, B):
        """one cycle from x = 0 per column; column j == vcycle(B[j])"""
        X = [self._new_own(0) for _ in B]
        bp, k1 = self._vecs_multi(B)
        xp, k2 = self._vecs_multi(X, writable=True)
        self._ck(self.lib.pamg_vcycle_multi(self._h, len(B), bp, xp))
        return X

    def pcg_multi(self, B, rtol=1e-8, maxiter=200, mode=1):
        """k independent solves (mode 0 CG, 1 AMG-PCG, 2 flexible); per column the results tuple of pcg():
        list of (x, iters, hist, converged), column j == pcg(B[j]) (mode 0/1) or fcg(B[j]) (mode 2)"""
        k = len(B)
        X = [self._new_own(0) for _ in B]
        bp, k1 = self._vecs_multi(B)
        xp, k2 = self._vecs_multi(X, writable=True)
        it = np.zeros(k, np.int32)
        conv = np.zeros(k, np.int32)
        hist = np.zeros((k, maxiter + 1))
        self._ck(self.lib.pamg_pcg_multi(self._h, k, bp, xp, float(rtol), int(maxiter), int(mode), _ptr(it, C.c_int32),
                                         _ptr(conv, C.c_int32), _ptr(hist, C.c_double)), allow=(ERR_NOTCONV,))
        return [(X[j], int(it[j]), hist[j, :it[j] + 1].copy(), bool(conv[j])) for j in range(k)]

    def time_kernel_multi(self, k, kind, level, reps=10, flush_l2=True):
        """time_kernel over k columns: one k-wide launch where the block has one, else k single launches"""
        ms = np.zeros(reps, np.float32)
        self._ck(self.lib.pamg_time_kernel_multi(self._h, int(k), kind, level, reps, int(flush_l2), _ptr(ms, C.c_float)))
        return ms

    def load_rhs(self, b):
        bp, k1 = self._vecs(b)
        self._ck(self.lib.pamg_load_rhs(self._h, bp))

    def pcg_resident(self, rtol=1e-8, maxiter=200, precond=True):
        it = C.c_int32()
        hist = np.zeros(maxiter + 2)
        st = self._ck(self.lib.pamg_pcg_resident(self._h, float(rtol), int(maxiter), int(bool(precond)), C.byref(it),
                                                 _ptr(hist, C.c_double)), allow=(ERR_NOTCONV,))
        return it.value, hist[:it.value + 1].copy(), st == OK

    def read_solution(self):
        x = self._new_own(0)
        xp, k = self._vecs(x, writable=True)
        self._ck(self.lib.pamg_read_solution(self._h, xp))
        return x

    def time_kernel(self, kind, level, reps=10, flush_l2=True):
        ms = np.zeros(reps, np.float32)
        self._ck(self.lib.pamg_time_kernel(self._h, kind, level, reps, int(flush_l2), _ptr(ms, C.c_float)))
        return ms

    def trace_enable(self, capacity=1 << 16):
        self._ck(self.lib.pamg_trace_enable(self._h, int(capacity)))

    def trace_read(self, part, cap=1 << 16):
        out = np.zeros(cap, np.uint64)
        n = C.c_int32()
        self._ck(self.lib.pamg_trace_read(self._h, int(part), _ptr(out, C.c_uint64), cap, C.byref(n)))
        return out[:n.value].copy()

    def trace_names(self):
        buf = C.create_string_buffer(1 << 16)
        self._ck(self.lib.pamg_trace_names(self._h, buf, len(buf)))
        return [s for s in buf.value.decode().split("\n") if s]

    def stats(self):
        s = Stats()
        self._ck(self.lib.pamg_get_stats(self._h, C.byref(s)))
        return s
