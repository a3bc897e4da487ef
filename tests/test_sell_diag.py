"""SELL with implied columns (csrc/formats.hpp diag_layout, kernels.cuh k_spmv_sell_diag).

Stencil operators store one value-index byte per (row, offset) slot and no column: the column of slot j is row + off[j].  The
layout is built by the same host function the upload uses and queried through pamg_layout_sell_diag, so it is checked here
without a GPU: every stored entry reconstructs the own-own CSR block exactly (column, value bits, order), and the blocks that
must not take the layout report ndiag = 0.  The GPU tests run the new kernel against the column-stored value-indexed SELL
kernel it replaces (same bits) and against the oracle."""
import functools

import numpy as np
import pytest
import scipy.sparse as sp

import amg_oracle as O
from parallel_amg_b200 import _lib as L
from util import det_vector, own_parts, product_context_from_oracle, rel_err

ABSENT = 255


def _context(kind, dims, pp, **opts):
    c = L.Context(int(np.prod(pp)))
    if kind == "poisson":
        c.gallery_poisson(dims, pp)
    elif kind == "jump":
        c.gallery_diffusion_jump(dims, pp, blocks=8, kmax=1.0e4, eps_z=1.0e-3)
    else:
        c.gallery_elasticity(dims, pp)
    c.setup(c.default_options(**opts))
    return c


def _reconstruct(lay, nrows):
    """CSR (indptr, indices, data) of the slots that hold an entry, rows in order, slots by ascending offset."""
    off, d, idx = lay["off"], lay["dict"], lay["idx"]
    nd = len(off)
    ns = (nrows + 127) // 128
    assert len(idx) == ns * nd * 128
    code = idx.reshape(ns, nd, 128)
    q = np.arange(128)
    rows = np.empty((ns, 128), np.int64)
    for sl in range(ns):
        base = sl * 128
        rows[sl] = base + ((q % 4) * 32 + q // 4 if base + 128 <= nrows else q)   # byte 4 lane + k <-> row 32 k + lane (full slice)
    row_of = np.broadcast_to(rows[:, None, :], code.shape)
    j_of = np.broadcast_to(np.arange(nd)[None, :, None], code.shape)
    live = code != ABSENT
    assert np.all(row_of[live] < nrows)                   # the tail of the last slice holds nothing
    r, j, k = row_of[live], j_of[live], code[live]
    order = np.lexsort((j, r))
    r, j, k = r[order], j[order], k[order]
    cols = r + off[j]
    indptr = np.zeros(nrows + 1, np.int64)
    np.add.at(indptr, r + 1, 1)
    return np.cumsum(indptr), cols, d[k]


ROUND_TRIP = [("poisson", (40, 37), (1, 1)), ("poisson", (40, 37), (2, 2)), ("poisson", (17, 15, 13), (1, 1, 1)),
              ("poisson", (17, 15, 13), (2, 2, 1)), ("poisson", (33, 31, 17), (3, 2, 1)), ("jump", (24, 24, 24), (1, 1, 1)),
              ("jump", (24, 20, 18), (2, 2, 2))]


@pytest.mark.parametrize("kind,dims,pp", ROUND_TRIP, ids=[f"{k}-{'x'.join(map(str, d))}-p{int(np.prod(p))}" for k, d, p in ROUND_TRIP])
def test_layout_round_trip(kind, dims, pp):
    c = _context(kind, dims, pp)
    for p in range(c.nparts):
        ip, ix, val = c.block(0, p, L.A_OO)
        nr = len(ip) - 1
        lay = c.layout_sell_diag(0, p)
        assert lay is not None, "a stencil block must take the diagonal layout"
        off = lay["off"]
        assert 1 <= len(off) <= (5 if len(dims) == 2 else 7) and np.all(np.diff(off) > 0)
        assert len(off) * nr <= 1.25 * len(ix)
        rp, rc, rv = _reconstruct(lay, nr)
        assert np.array_equal(rp, ip)                                           # absent slots = exactly the missing entries
        assert np.array_equal(rc, ix)                                           # column = row + off, stored order
        assert np.array_equal(rv.view(np.uint64), val.view(np.uint64))          # dict[idx] == val bit for bit
        vi = c.layout_sell_values(0, p, L.A_OO, 128, -4)                        # the dictionary of the value-indexed layouts, unchanged
        assert vi is not None and np.array_equal(vi[0][:256].view(np.uint64), lay["dict"].view(np.uint64))


def test_refused_elasticity_and_coarse_levels():
    c = _context("elasticity", (6, 6, 6), (1, 1, 1), coarse_size=40)
    assert c.layout_sell_diag(0, 0) is None                                     # 81 entries per row over ~135 offsets
    c = _context("poisson", (24, 24, 24), (2, 1, 1), coarse_size=40)
    assert c.num_levels() >= 3
    for p in range(2):
        assert c.layout_sell_diag(0, p) is not None
        assert c.layout_sell_diag(1, p) is None                                 # the Galerkin operator: irregular columns
        assert c.layout_sell_diag(0, p, L.P_OO) is None and c.layout_sell_diag(0, p, L.R_OO) is None


def _single_block(A):
    """A one-level hierarchy whose level-0 own-own block is A exactly as given (entry order included)."""
    n = A.shape[0]
    c = L.Context(1)
    e64, e32 = np.zeros(0, np.int64), np.zeros(0, np.int32)
    lev = dict(own_to_global=np.arange(n, dtype=np.int64), ghost_to_global=e64, ghost_to_owner=e32, A_oo=A)
    c.upload_hierarchy([[lev]], np.linalg.inv(A.toarray()), c.default_options())
    return c


def _tridiag(n, lower, diag, upper):
    i = np.arange(n - 1)
    return sp.csr_matrix(sp.coo_matrix((np.concatenate([lower, diag, upper]),
                                        (np.concatenate([i + 1, np.arange(n), i]), np.concatenate([i, np.arange(n), i + 1]))),
                                       shape=(n, n)))


def test_refused_unsorted_row():
    A = _tridiag(300, -np.ones(299), np.full(300, 4.0), -np.ones(299))
    A.sort_indices()
    assert _single_block(A).layout_sell_diag(0, 0) is not None
    A.indices[A.indptr[100]:A.indptr[101]] = A.indices[A.indptr[100]:A.indptr[101]][::-1].copy()   # row 100: 101, 100, 99
    A.data[A.indptr[100]:A.indptr[101]] = A.data[A.indptr[100]:A.indptr[101]][::-1].copy()
    assert _single_block(A).layout_sell_diag(0, 0) is None


@pytest.mark.parametrize("ndist,ok", [(254, True), (255, False), (256, False)])
def test_refused_too_many_values(ndist, ok):
    """One code (255) marks an absent slot, so at most 254 distinct non-zero values fit."""
    n = 600
    vals = 1.0 + np.arange(n - 1) % (ndist - 1)                                # ndist - 1 off-diagonal values + the diagonal
    A = _tridiag(n, -vals, np.full(n, 1000.0), -vals)
    A.sort_indices()
    lay = _single_block(A).layout_sell_diag(0, 0)
    assert (lay is not None) == ok
    if ok:
        rp, rc, rv = _reconstruct(lay, n)
        assert np.array_equal(rc, A.indices) and np.array_equal(rv, A.data)


def test_refused_fill_above_limit():
    n = 600
    A = sp.lil_matrix((n, n))
    A.setdiag(4.0)
    for k in range(1, 11):                                                      # ten rows with one far entry each, ten offsets
        A[k, k + 50 * k] = -1.0
        A[k + 50 * k, k] = -1.0
    A = sp.csr_matrix(A)
    A.sort_indices()
    assert 21 * n > 1.25 * A.nnz
    assert _single_block(A).layout_sell_diag(0, 0) is None


# ---- GPU: the new kernel against the column-stored value-indexed kernel, bit for bit ----------------------------------------------
@functools.lru_cache(maxsize=8)
def _oracle(kind, dims, pp, smoother):
    A = O.poisson_fd(dims) if kind == "poisson" else O.diffusion_fv(dims, O.jump_coefficient_k(dims))
    owner = O.uniform_partition(pp, dims)
    oopts = {"smoother": smoother} if smoother != "jacobi" else {}
    if kind == "jump":
        oopts["eps_strength"] = 0.08                                            # config 5's filtered strength (as in test_gpu_parity_at_size)
    return A, O.build(A, owner, int(np.prod(pp)), oopts), oopts


GPU_CASES = [("poisson", (28, 28, 28), (1, 1, 1)), ("poisson", (33, 31, 17), (3, 2, 1)), ("poisson", (200, 200), (2, 2)),
             ("jump", (24, 24, 24), (2, 2, 2))]


@pytest.mark.gpu
@pytest.mark.parametrize("smoother", ["jacobi", "l1jacobi", "chebyshev"])
@pytest.mark.parametrize("kind,dims,pp", GPU_CASES, ids=[f"{k}-{'x'.join(map(str, d))}-p{int(np.prod(p))}" for k, d, p in GPU_CASES])
def test_sell_diag_is_bit_identical_to_sell(kind, dims, pp, smoother):
    A, h, oopts = _oracle(kind, dims, pp, smoother)
    cd = product_context_from_oracle(h, oopts, spmv_format=L.FORMAT_SELL_DIAG)
    cd.device_init()
    cs = product_context_from_oracle(h, oopts, spmv_format=L.FORMAT_SELL)
    cs.device_init()
    vd, vs = cd.stats().value_indexed, cs.stats().value_indexed
    assert vd[0] & 64 and not vs[0] & 64 and vd[0] & ~64 == vs[0], (vd[0], vs[0])   # level 0 of A takes the layout, only under SELL_DIAG
    assert not vd[1] & 64 and cd.stats().format[0] == L.FORMAT_SELL
    lev = h["levels"][0]
    n = A.shape[0]
    b_, x_ = det_vector(n, 41), det_vector(n, 42)
    for a, b in zip(cd.spmv(0, own_parts(lev, x_)), cs.spmv(0, own_parts(lev, x_))):
        assert np.array_equal(a, b)
    ra, rb = cd.residual_restrict(0, own_parts(lev, b_), own_parts(lev, x_)), cs.residual_restrict(0, own_parts(lev, b_), own_parts(lev, x_))
    for a, b in zip(ra[0] + ra[1], rb[0] + rb[1]):
        assert np.array_equal(a, b)
    for a, b in zip(cd.smooth(0, 2, own_parts(lev, b_), own_parts(lev, x_)), cs.smooth(0, 2, own_parts(lev, b_), own_parts(lev, x_))):
        assert np.array_equal(a, b)
    rhs = A @ det_vector(n, 17)
    for a, b in zip(cd.vcycle(own_parts(lev, rhs)), cs.vcycle(own_parts(lev, rhs))):
        assert np.array_equal(a, b)
    (x, it, hist, ok), (x0, it0, hist0, ok0) = cd.pcg(own_parts(lev, rhs)), cs.pcg(own_parts(lev, rhs))
    assert ok == ok0 and it == it0
    assert np.array_equal(hist, hist0)                                          # same grid: the fused dots add in the same order
    for a, b in zip(x, x0):
        assert np.array_equal(a, b)
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, rhs))
    assert it == it_ref
    if it < 100:   # l1-Jacobi on the 8-part jump problem needs 199 steps; over that many the history drifts from the oracle beyond 1e-7 in both formats
        assert np.allclose(hist, hist_ref, rtol=1e-7)
    cd.close()
    cs.close()


@pytest.mark.gpu
@pytest.mark.timeout(600, method="thread")
@pytest.mark.parametrize("kind,dims,pp", [("poisson", (64, 64, 64), (1, 1, 1)), ("poisson", (128, 128, 128), (2, 1, 1)),
                                          ("elasticity", (42, 42, 42), (1, 1, 1))], ids=["poisson-64-p1", "poisson-128-p2", "elasticity-42-p1"])
def test_auto_takes_the_layout_for_stencils_only(kind, dims, pp):
    c = _context(kind, dims, pp)
    c.device_init()
    vi = list(c.stats().value_indexed)
    if kind == "elasticity":
        assert not any(v & 64 for v in vi)
    else:
        assert vi[0] & 64 and not any(v & 64 for v in vi[1:])
        assert c.stats().format[0] == L.FORMAT_SELL
    n, _ = c.global_size()
    own = [c.index_maps(0, p)[0] for p in range(c.nparts)]
    rhs = c.host_matvec_global(det_vector(n, 1))
    x1, it1, h1, ok1 = c.pcg([rhs[o] for o in own], rtol=1e-8, maxiter=400)
    x2, it2, h2, ok2 = c.pcg([rhs[o] for o in own], rtol=1e-8, maxiter=400)   # the second solve replays the captured graph
    assert ok1 and ok2 and it1 == it2 and np.array_equal(h1, h2)
    for a, b in zip(x1, x2):
        assert np.array_equal(a, b)
    c.close()
