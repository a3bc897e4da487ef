"""Several right-hand sides per pass over the hierarchy (pamg_spmv_multi / pamg_vcycle_multi / pamg_pcg_multi).

The contract is bit-identity per column: column j of every multi call equals the single-vector call on column j alone (the
same hierarchy and kernel options; on one GPU the single call runs exactly the split halo protocol the multi calls use).  The
k-wide kernels (k_spmv_sell_diag_multi, k_spmv_sell_vi4_multi) keep the single kernels' slice map, grid, per-row product order and
epilogue, so the comparisons below are np.array_equal, never a tolerance.  Without a GPU: argument checks through the ABI and the
register budget of the new kernels."""
import os
import re

import numpy as np
import pytest

from parallel_amg_b200 import _lib as L
from util import det_vector

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KS = (1, 2, 3, 4, 5, 8)


def _context(kind, dims, pp, kmax=8, init=True, **opts):
    c = L.Context(int(np.prod(pp)))
    if kind == "poisson":
        c.gallery_poisson(dims, pp)
    elif kind == "jump":
        c.gallery_diffusion_jump(dims, pp, blocks=8, kmax=1.0e4, eps_z=1.0e-3)
    else:
        c.gallery_elasticity(dims, pp)
    c.setup(c.default_options(**opts))
    c.set_rhs_capacity(kmax)
    if init:
        c.device_init()
    return c


def _columns(c, level, k, seed0=1):
    return [[det_vector(c.level_info(level, p).n_own, seed=seed0 + 7 * j + p) for p in range(c.nparts)] for j in range(k)]


def _same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


# ---- no GPU -------------------------------------------------------------------------------------------------------------------------
def test_capacity_and_k_are_checked():
    c = _context("poisson", (6, 5, 4), (1, 1, 1), init=False)
    for bad in (0, 9, -1):
        with pytest.raises(L.PamgError) as e:
            c.set_rhs_capacity(bad)
        assert e.value.status == L.ERR_ARG and "capacity" in str(e.value)
    c.set_rhs_capacity(2)
    X = _columns(c, 0, 3)
    Y = [[np.zeros_like(v) for v in x] for x in X]

    def refused(call, k, text):
        xp, k1 = c._vecs_multi(X[:max(k, 1)])
        yp, k2 = c._vecs_multi(Y[:max(k, 1)], writable=True)
        assert call(k, xp, yp) == L.ERR_ARG
        assert text in c.lib.pamg_last_error(c._h).decode()

    spmv = lambda k, xp, yp: c.lib.pamg_spmv_multi(c._h, 0, k, xp, yp)
    vcyc = lambda k, xp, yp: c.lib.pamg_vcycle_multi(c._h, k, xp, yp)
    pcg = lambda k, xp, yp: c.lib.pamg_pcg_multi(c._h, k, xp, yp, 1e-8, 10, 1, None, None, None)
    for call in (spmv, vcyc, pcg):
        refused(call, 3, "capacity")  # k above the capacity: refused before any device state is touched
        refused(call, 0, "capacity")
        refused(call, 2, "pamg_device_init")  # no device state yet


def test_k_wide_kernels_do_not_spill():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    from ptxas_table import table
    rows = [r for r in table() if "_multi<" in r[0]]
    # diag and vi4 (one- and two-byte indices) x K in {2, 4} x 8 mode/dot instantiations
    assert len(rows) == 48, len(rows)
    for name, regs, spill, stack, smem in rows:
        assert spill == 0, (name, spill)
        assert regs <= 128, (name, regs)  # two CTAs per SM


# ---- GPU: spmv_multi ------------------------------------------------------------------------------------------------------------
SPMV_CASES = [("poisson", (20, 18, 16), (1, 1, 1), L.FORMAT_SELL_DIAG), ("poisson", (20, 18, 16), (2, 2, 1), L.FORMAT_SELL_DIAG),
              ("jump", (16, 16, 16), (1, 1, 1), L.FORMAT_SELL_DIAG), ("jump", (16, 16, 16), (2, 1, 2), L.FORMAT_SELL_DIAG),
              ("elasticity", (8, 8, 8), (1, 1, 1), L.FORMAT_SELL), ("elasticity", (8, 8, 8), (2, 1, 1), L.FORMAT_SELL),
              ("poisson", (20, 18, 16), (1, 1, 1), L.FORMAT_SELL), ("poisson", (20, 18, 16), (2, 2, 1), L.FORMAT_SELL)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,dims,pp,fmt", SPMV_CASES, ids=[f"{k}-{'x'.join(map(str, pp))}-f{f}" for k, d, pp, f in SPMV_CASES])
def test_spmv_multi_matches_spmv(kind, dims, pp, fmt):
    c = _context(kind, dims, pp, spmv_format=fmt)
    vi = [c.stats().value_indexed[l] for l in range(c.num_levels())]
    assert vi[0] & 1, vi  # level-0 A runs a kernel with a k-wide form
    for level in range(c.num_levels()):
        X = _columns(c, level, max(KS), seed0=3 + level)
        ref = [c.spmv(level, x) for x in X]
        for k in KS:
            got = c.spmv_multi(level, X[:k])
            for j in range(k):
                assert _same(got[j], ref[j]), (kind, pp, level, k, j)


def _synthetic(name, n, monkeypatch):
    from test_kernel_rows import case, product_context_from_oracle
    s = case(name, n)
    for k, v in s["env"].items():
        monkeypatch.setenv(k, v)
    c = product_context_from_oracle(s["h"], None, **s["opts"])
    c.set_rhs_capacity(8)
    c.device_init()
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["diag-7-40", "vi4-255", "vi4-256"])
@pytest.mark.parametrize("n", [1, 127, 128, 129, 4097])
def test_spmv_multi_ragged_rows(name, n, monkeypatch):
    c = _synthetic(name, n, monkeypatch)
    for level in range(c.num_levels()):
        X = _columns(c, level, 8, seed0=11)
        ref = [c.spmv(level, x) for x in X]
        for k in KS:
            got = c.spmv_multi(level, X[:k])
            assert all(_same(got[j], ref[j]) for j in range(k)), (name, n, level, k)


# ---- GPU: vcycle_multi ----------------------------------------------------------------------------------------------------------
VC = [(sm, cy, tr) for sm in (L.SMOOTHER_JACOBI, L.SMOOTHER_L1JACOBI, L.SMOOTHER_CHEBYSHEV) for cy in (L.CYCLE_V, L.CYCLE_W)
      for tr in (0, 600, None)]


@pytest.mark.gpu
@pytest.mark.parametrize("smoother,cycle,tail_rows", VC, ids=[f"s{a}-c{b}-t{c}" for a, b, c in VC])
def test_vcycle_multi_matches_vcycle(smoother, cycle, tail_rows):
    opts = dict(smoother=smoother, cycle=cycle, spmv_format=L.FORMAT_SELL_DIAG)
    if tail_rows is not None:
        opts["tail_rows"] = tail_rows
    c = _context("poisson", (24, 22, 20), (2, 2, 1), kmax=4, **opts)
    B = _columns(c, 0, 4, seed0=5)
    ref = [c.vcycle(b) for b in B]
    for k in (1, 3, 4):
        got = c.vcycle_multi(B[:k])
        assert all(_same(got[j], ref[j]) for j in range(k)), k
    got = c.vcycle_multi(B)  # graph replay
    assert all(_same(got[j], ref[j]) for j in range(4))


# ---- GPU: pcg_multi -------------------------------------------------------------------------------------------------------------
def _rhs_set(c):
    """columns that converge at different iterations: seeded, scaled by 1e6, zero, and a repeat of the first"""
    B = _columns(c, 0, 3, seed0=21)
    B[1] = [1.0e6 * v for v in B[1]]
    B.insert(2, [np.zeros_like(v) for v in B[0]])
    B.append([v.copy() for v in B[0]])
    return B


def _single(c, b, mode, rtol, maxiter):
    if mode == 2:
        return c.fcg(b, rtol=rtol, maxiter=maxiter)
    return c.pcg(b, rtol=rtol, maxiter=maxiter, precond=mode == 1)


def _assert_columns(got, ref, what):
    for j, (g, r) in enumerate(zip(got, ref)):
        assert g[1] == r[1], (what, j, g[1], r[1])
        assert g[3] == r[3], (what, j)
        assert np.array_equal(g[2], r[2]), (what, j)
        assert _same(g[0], r[0]), (what, j)


PCG_CASES = [("poisson", (24, 22, 20), (1, 1, 1), L.FORMAT_SELL_DIAG), ("poisson", (24, 22, 20), (2, 2, 1), L.FORMAT_SELL_DIAG),
             ("elasticity", (9, 8, 8), (1, 1, 1), L.FORMAT_SELL)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("kind,dims,pp,fmt", PCG_CASES, ids=[f"{k}-{'x'.join(map(str, pp))}" for k, d, pp, f in PCG_CASES])
def test_pcg_multi_matches_pcg(kind, dims, pp, fmt, mode):
    c = _context(kind, dims, pp, kmax=8, spmv_format=fmt)
    B = _rhs_set(c)
    ref = [_single(c, b, mode, 1e-8, 400) for b in B]
    assert ref[2][1] == 0 and all(np.all(v == 0) for v in ref[2][0])  # zero column: no iteration, x = 0
    assert len({r[1] for r in ref}) >= 2  # the columns stop at different iterations
    got = c.pcg_multi(B, rtol=1e-8, maxiter=400, mode=mode)
    _assert_columns(got, ref, "first call")
    st = c.stats()
    assert st.iters == max(r[1] for r in ref)
    _assert_columns(c.pcg_multi(B, rtol=1e-8, maxiter=400, mode=mode), ref, "graph replay")
    _assert_columns(c.pcg_multi(B[:1], rtol=1e-8, maxiter=400, mode=mode), ref[:1], "k = 1")
    # a maxiter that truncates some columns
    short = max(2, min(r[1] for r in ref if r[1] > 0) - 1)
    ref_s = [_single(c, b, mode, 1e-8, short) for b in B]
    assert not all(r[3] for r in ref_s)
    _assert_columns(c.pcg_multi(B, rtol=1e-8, maxiter=short, mode=mode), ref_s, "truncated")
    # without graphs: the same bits
    c.set_kernel_options(use_graph=0, spmv_format=fmt)
    c.device_init()
    _assert_columns(c.pcg_multi(B, rtol=1e-8, maxiter=400, mode=mode), ref, "use_graph = 0")


@pytest.mark.gpu
def test_pcg_multi_status_code():
    c = _context("poisson", (16, 16, 16), (1, 1, 1), kmax=2, spmv_format=L.FORMAT_SELL_DIAG)
    B = _columns(c, 0, 2)
    X = [c._new_own(0) for _ in B]
    bp, k1 = c._vecs_multi(B)
    xp, k2 = c._vecs_multi(X, writable=True)
    it = np.zeros(2, np.int32)
    conv = np.zeros(2, np.int32)
    st = c.lib.pamg_pcg_multi(c._h, 2, bp, xp, 1e-10, 3, 1, it.ctypes.data_as(L.C.POINTER(L.C.c_int32)),
                              conv.ctypes.data_as(L.C.POINTER(L.C.c_int32)), None)
    assert st == L.ERR_NOTCONV and list(conv) == [0, 0] and list(it) == [3, 3]
    st = c.lib.pamg_pcg_multi(c._h, 2, bp, xp, 1e-8, 400, 1, it.ctypes.data_as(L.C.POINTER(L.C.c_int32)),
                              conv.ctypes.data_as(L.C.POINTER(L.C.c_int32)), None)
    assert st == L.OK and list(conv) == [1, 1]


@pytest.mark.gpu
def test_capacity_change_needs_device_init():
    c = _context("poisson", (12, 12, 12), (1, 1, 1), kmax=2)
    B = _columns(c, 0, 2)
    c.vcycle_multi(B)
    c.set_rhs_capacity(4)
    with pytest.raises(L.PamgError) as e:
        c.vcycle_multi(B)
    assert e.value.status == L.ERR_ARG and "pamg_device_init" in str(e.value)
    c.device_init()
    c.vcycle_multi(B + B)


@pytest.mark.gpu
def test_trace_names_show_k_wide_launches():
    c = _context("poisson", (40, 40, 40), (1, 1, 1), kmax=4, spmv_format=L.FORMAT_SELL)
    c.pcg_multi(_columns(c, 0, 4), rtol=1e-8, maxiter=50, mode=1)
    names = c.trace_names()
    for block in ("A0", "R0", "A1"):  # P keeps its single launches (engine.cu multi_width)
        assert any(re.match(rf"sell-vi(16)? x4 \S+ {block}\b", n) for n in names), (block, names)


# ---- GPU: configuration sizes, AUTO formats ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.timeout(900, method="thread")
@pytest.mark.parametrize("kind,dims", [("poisson", (128, 128, 128)), ("elasticity", (42, 42, 42))])
def test_pcg_multi_at_size(kind, dims):
    c = _context(kind, dims, (1, 1, 1), kmax=4)
    B = _columns(c, 0, 4, seed0=31)
    ref = [c.pcg(b, rtol=1e-8, maxiter=500) for b in B]
    got = c.pcg_multi(B, rtol=1e-8, maxiter=500, mode=1)
    _assert_columns(got, ref, kind)
    assert any(" x4 " in n and n.endswith("A0") for n in c.trace_names())
