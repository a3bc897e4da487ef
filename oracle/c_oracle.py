"""ctypes front-end of oracle/pamg_oracle.c (the C + OpenMP restatement of the solve phase).
TEST INFRASTRUCTURE ONLY — see the header of pamg_oracle.c.  PARITY UNPINNED (no reference code).

Built with plain gcc into oracle/_build/ (git-ignored, travels to the GPU box)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pamg_oracle.c")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libpamg_oracle.so")
STAMP = os.path.join(OUT_DIR, "libpamg_oracle.stamp")
FLAGS = ["-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-std=c11"]


def _digest():
    with open(SRC, "rb") as fh:
        return hashlib.sha256(fh.read() + " ".join(FLAGS).encode()).hexdigest()


def build(force=False):
    # Rebuild on a change of the source or flags, not of mtimes: a copied tree keeps a valid library and may be read-only.
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig:
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    r = subprocess.run(["gcc"] + FLAGS + [SRC, "-o", LIB, "-lm"], capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError("gcc failed:\n" + r.stderr)
    with open(STAMP, "w") as fh:
        fh.write(dig)
    return LIB


_i64p, _i32p, _f64p = C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_double)


def _load():
    lib = C.CDLL(build())
    lib.orc_create.restype = C.c_void_p
    lib.orc_create.argtypes = [C.c_int32] * 4
    lib.orc_set_part.restype = None
    lib.orc_set_part.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.POINTER(_i64p),
                                 C.POINTER(_i32p), C.POINTER(_f64p), _f64p, _i32p, _i32p]
    lib.orc_set_coarse.restype = None
    lib.orc_set_coarse.argtypes = [C.c_void_p, C.c_int64, _f64p, C.c_int32, _i64p, _i64p]
    lib.orc_destroy.restype = None
    lib.orc_destroy.argtypes = [C.c_void_p]
    lib.orc_set_cycle.restype = None
    lib.orc_set_cycle.argtypes = [C.c_void_p, C.c_int32]
    lib.orc_vcycle.restype = None
    lib.orc_vcycle.argtypes = [C.c_void_p, C.POINTER(_f64p), C.POINTER(_f64p)]
    lib.orc_pcg.restype = C.c_int32
    lib.orc_pcg.argtypes = [C.c_void_p, C.POINTER(_f64p), C.POINTER(_f64p), C.c_double, C.c_int32, C.c_int32, _f64p]
    lib.orc_fgmres.restype = C.c_int32
    lib.orc_fgmres.argtypes = [C.c_void_p, C.POINTER(_f64p), C.POINTER(_f64p), C.c_double, C.c_int32, C.c_int32, C.c_int32, _f64p]
    return lib


def _p(a, ct):
    return a.ctypes.data_as(C.POINTER(ct))


class COracle:
    """levels[l][p]: dict with own_to_global, ghost_to_global, ghost_to_owner, blocks
    'A_oo','A_og'[, 'P_oo','P_og','R_oo','R_og'] as objects with .indptr/.indices/.data, and 'w'
    (smoother weight per own row: omega/a_ii for Jacobi, 1/l1-diag for l1-Jacobi)."""

    NAMES = ("A_oo", "A_og", "P_oo", "P_og", "R_oo", "R_og")

    def __init__(self, levels, coarse_inv, nu_pre=1, nu_post=1, cycle="v"):
        self.lib = _load()
        self.nparts = len(levels[0])
        self.L = len(levels)
        self.keep = []
        self.h = self.lib.orc_create(self.nparts, self.L, nu_pre, nu_post)
        self.lib.orc_set_cycle(self.h, 1 if cycle == "w" else 0)
        self.n_own = [[len(d["own_to_global"]) for d in lev] for lev in levels]
        for l, lev in enumerate(levels):
            for p, d in enumerate(lev):
                own = np.ascontiguousarray(d["own_to_global"], np.int64)
                gh = np.ascontiguousarray(d["ghost_to_global"], np.int64)
                gho = np.ascontiguousarray(d["ghost_to_owner"], np.int32)
                lid = np.zeros(len(gh), np.int32)
                for q in np.unique(gho):
                    sel = gho == q
                    oq = np.asarray(levels[l][int(q)]["own_to_global"], np.int64)
                    pos = np.searchsorted(oq, gh[sel])
                    assert np.array_equal(oq[pos], gh[sel])
                    lid[sel] = pos
                ptr = (_i64p * 6)()
                col = (_i32p * 6)()
                val = (_f64p * 6)()
                for b, name in enumerate(self.NAMES):
                    m = d.get(name)
                    if m is None:
                        continue
                    ip = np.ascontiguousarray(m.indptr, np.int64)
                    ix = np.ascontiguousarray(m.indices, np.int32)
                    dd = np.ascontiguousarray(m.data, np.float64)
                    self.keep += [ip, ix, dd]
                    ptr[b], col[b], val[b] = _p(ip, C.c_int64), _p(ix, C.c_int32), _p(dd, C.c_double)
                w = np.ascontiguousarray(d["w"], np.float64)
                self.keep += [own, gh, gho, lid, w]
                n_own_c = len(levels[l + 1][p]["own_to_global"]) if l + 1 < self.L else 0
                self.lib.orc_set_part(self.h, l, p, len(own), len(gh), n_own_c, ptr, col, val, _p(w, C.c_double),
                                      _p(gho, C.c_int32), _p(lid, C.c_int32))
                if l == self.L - 1:
                    inv = np.ascontiguousarray(coarse_inv, np.float64)
                    self.keep.append(inv)
                    self.lib.orc_set_coarse(self.h, inv.shape[0], _p(inv, C.c_double), p, _p(own, C.c_int64), _p(gh, C.c_int64))

    @classmethod
    def from_oracle_hierarchy(cls, h):
        import amg_oracle as O
        levels = []
        for lev in h["levels"]:
            parts = []
            for d in lev["parts"]:
                e = dict(d)
                e["w"] = O._wdinv(d, h["opts"])
                parts.append(e)
            levels.append(parts)
        return cls(levels, h["coarse_inv"], h["opts"]["nu_pre"], h["opts"]["nu_post"], h["opts"].get("cycle", "v"))

    @classmethod
    def from_product_context(cls, ctx, nparts, nu_pre=1, nu_post=1, omega=2.0 / 3.0, smoother="jacobi", cycle="v"):
        """The hierarchy the PRODUCT's host setup built, copied out through the C ABI queries (pamg_get_index_maps /
        pamg_get_block / pamg_get_diag / pamg_get_coarse_inverse), so that the oracle and the device run the same
        operators at sizes where the numpy oracle's own setup would take minutes.  ctx: parallel_amg_b200._lib.Context."""
        from types import SimpleNamespace
        nl = ctx.num_levels()
        levels = []
        for l in range(nl):
            parts = []
            for p in range(nparts):
                own, gh, gho = ctx.index_maps(l, p)
                d = dict(own_to_global=own, ghost_to_global=gh, ghost_to_owner=gho)
                for b, name in enumerate(cls.NAMES):
                    if l == nl - 1 and b >= 2:
                        continue
                    ip, ix, dd = ctx.block(l, p, b)
                    d[name] = SimpleNamespace(indptr=ip, indices=ix, data=dd)
                dg, dl1 = ctx.diag(l, p)
                d["w"] = (1.0 / dl1) if smoother == "l1jacobi" else omega / dg
                parts.append(d)
            levels.append(parts)
        return cls(levels, ctx.coarse_inverse(), nu_pre, nu_post, cycle)

    def _vecs(self, arrs):
        out = (_f64p * self.nparts)()
        keep = [np.ascontiguousarray(a, np.float64) for a in arrs]
        for p, a in enumerate(keep):
            out[p] = _p(a, C.c_double)
        return out, keep

    def vcycle(self, b_parts):
        z = [np.zeros(n) for n in self.n_own[0]]
        bp, k1 = self._vecs(b_parts)
        zp, k2 = self._vecs(z)
        self.lib.orc_vcycle(self.h, bp, zp)
        return k2

    def pcg(self, b_parts, rtol=1e-8, maxiter=200, precond=True, flexible=False):
        x = [np.zeros(n) for n in self.n_own[0]]
        bp, k1 = self._vecs(b_parts)
        xp, k2 = self._vecs(x)
        hist = np.zeros(maxiter + 2)
        mode = 2 if (flexible and precond) else int(bool(precond))
        it = self.lib.orc_pcg(self.h, bp, xp, float(rtol), int(maxiter), mode, _p(hist, C.c_double))
        return k2, int(it), hist[: it + 1].copy()

    def fgmres(self, b_parts, rtol=1e-8, maxiter=200, restart=30, precond=True):
        x = [np.zeros(n) for n in self.n_own[0]]
        bp, k1 = self._vecs(b_parts)
        xp, k2 = self._vecs(x)
        hist = np.zeros(maxiter + 2)
        it = self.lib.orc_fgmres(self.h, bp, xp, float(rtol), int(maxiter), int(restart), int(bool(precond)), _p(hist, C.c_double))
        return k2, int(it), hist[: it + 1].copy()

    def close(self):
        if self.h:
            self.lib.orc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


if __name__ == "__main__":
    print(build(force=True))
