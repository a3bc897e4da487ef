"""GPU parity tests (run with -m gpu on the B200 box): every kernel, the V-cycle and PCG against
the oracle on the SAME operators (the oracle-built hierarchy is uploaded through
pamg_level_upload), through the C ABI.  fp64 tolerances are the ones BASELINE.json north_star
states: 1e-12 relative per V-cycle, identical PCG iteration counts at rtol 1e-8."""
import numpy as np
import pytest

import amg_oracle as O
from parallel_amg_b200 import _lib as L
from util import (det_vector, oracle_problem, own_of, own_parts, product_context_from_oracle, product_options, rel_err)

pytestmark = pytest.mark.gpu

TOL_KERNEL = 1e-13   # one SpMV-shaped pass
TOL_VCYCLE = 1e-12   # north_star: per V-cycle, fp64

# (dims, parts): 1 part = plain single GPU; >1 parts share cuda:0 (debug-backend layout)
PROBLEMS = [((20, 20, 20), (1, 1, 1)), ((20, 20, 20), (2, 2, 2)), ((33, 31, 17), (3, 2, 1)), ((200, 200), (2, 2))]


def make(dims, pp, oopts=None, **extra):
    A, owner, h = oracle_problem(dims, pp, tuple(sorted((oopts or {}).items())))
    c = product_context_from_oracle(h, oopts, **extra)
    c.device_init()
    return A, h, c


@pytest.mark.parametrize("dims,pp", PROBLEMS)
def test_spmv_every_level(dims, pp):
    A, h, c = make(dims, pp)
    for l, lev in enumerate(h["levels"]):
        n = h["global"]["levels"][l]["A"].shape[0]
        x = det_vector(n, 11 + l)
        ref = own_of(lev, O.spmv(lev, O.pvector_from_global(lev, x)))
        got = c.spmv(l, own_parts(lev, x))
        assert rel_err(got, ref) <= TOL_KERNEL


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
def test_spmv_all_lane_widths(lanes):
    A, h, c = make((20, 20, 20), (2, 1, 1), None, lanes_per_row=lanes, spmv_format=L.FORMAT_CSR)
    lev = h["levels"][0]
    x = det_vector(A.shape[0], 3)
    ref = own_of(lev, O.spmv(lev, O.pvector_from_global(lev, x)))
    assert rel_err(c.spmv(0, own_parts(lev, x)), ref) <= TOL_KERNEL
    assert c.stats().lanes[0] == lanes and c.stats().format[0] == L.FORMAT_CSR


FORMATS = {"csr": dict(spmv_format=L.FORMAT_CSR), "stream": dict(spmv_format=L.FORMAT_STREAM),
           "sell1": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=1, sell_sigma=1),
           "sell2": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=2),
           "sell2-sorted": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=2, sell_sigma=256),
           "sell1-sorted": dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=1, sell_sigma=96)}


@pytest.mark.parametrize("fmt", sorted(FORMATS))
def test_all_kernel_families_vcycle_and_pcg(fmt):
    """Every SpMV family (sub-warp CSR, CSR-stream, SELL-C-sigma with and without row sorting) must
    give the same answers: per-level operators, the V-cycle and the PCG iteration count."""
    A, h, c = make((33, 31, 17), (3, 2, 1), None, **FORMATS[fmt])
    f = FORMATS[fmt]["spmv_format"]
    assert c.stats().format[0] == f and c.stats().format_p[0] == f and c.stats().format_r[0] == f
    for l in range(len(h["levels"]) - 1):
        lev, nxt = h["levels"][l], h["levels"][l + 1]
        gl = h["global"]["levels"][l]
        n, nc = gl["A"].shape[0], h["global"]["levels"][l + 1]["A"].shape[0]
        b_, x_, ec = det_vector(n, 41), det_vector(n, 42), det_vector(nc, 43)
        assert rel_err(c.spmv(l, own_parts(lev, x_)), own_parts(lev, gl["A"] @ x_)) <= TOL_KERNEL
        r, bc = c.residual_restrict(l, own_parts(lev, b_), own_parts(lev, x_))
        assert rel_err(bc, own_parts(nxt, gl["R"] @ (b_ - gl["A"] @ x_))) <= 4 * TOL_KERNEL
        got = c.prolong_correct(l, own_parts(nxt, ec), own_parts(lev, x_))
        assert rel_err(got, own_parts(lev, x_ + gl["P"] @ ec)) <= TOL_KERNEL
    lev = h["levels"][0]
    b = det_vector(A.shape[0], 17)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, b))
    x, it, hist, ok = c.pcg(own_parts(lev, b))
    assert ok and it == it_ref and np.allclose(hist, hist_ref, rtol=1e-7)


@pytest.mark.parametrize("fmt", ["stream", "sell1", "sell2", "sell2-sorted"])
def test_spmv_is_bit_identical_to_sequential_row_sums(fmt):
    """The stream and SELL kernels round each product before adding them in column order, exactly like
    the oracle's C restatement (`s += a_ij * x_j`, no FMA): y must match bit for bit on one part."""
    A, h, c = make((28, 28, 28), (1, 1, 1), None, **FORMATS[fmt])
    x = det_vector(A.shape[0], 23)
    y = c.spmv(0, [x])[0]
    ref = np.zeros_like(x)
    Ac = A.tocsr()
    prod = Ac.data * x[Ac.indices]
    for k in range(7):  # column-ordered sequential sum, vectorised over rows
        idx = Ac.indptr[:-1] + k
        ok = idx < Ac.indptr[1:]
        ref[ok] = ref[ok] + prod[idx[ok]]
    assert np.array_equal(y, ref)


@pytest.mark.parametrize("dims,pp", PROBLEMS[:3])
@pytest.mark.parametrize("smoother", ["jacobi", "l1jacobi", "chebyshev"])
def test_smoother_sweeps(dims, pp, smoother):
    oopts = {"smoother": smoother}
    A, h, c = make(dims, pp, oopts)
    for l, lev in enumerate(h["levels"][:-1]):
        n = h["global"]["levels"][l]["A"].shape[0]
        b, x0 = det_vector(n, 21 + l), det_vector(n, 31 + l)
        for nu in (1, 2):
            ref = O.smooth(h, l, O.pvector_from_global(lev, x0), O.pvector_from_global(lev, b), nu)
            got = c.smooth(l, nu, own_parts(lev, b), own_parts(lev, x0))
            assert rel_err(got, own_of(lev, ref)) <= 4 * TOL_KERNEL


@pytest.mark.parametrize("dims,pp", PROBLEMS)
def test_residual_restrict_and_prolong_correct(dims, pp):
    A, h, c = make(dims, pp)
    for l in range(len(h["levels"]) - 1):
        lev, nxt = h["levels"][l], h["levels"][l + 1]
        n = h["global"]["levels"][l]["A"].shape[0]
        nc = h["global"]["levels"][l + 1]["A"].shape[0]
        b, x, ec = det_vector(n, 41), det_vector(n, 42), det_vector(nc, 43)
        gl = h["global"]["levels"][l]
        r_ref = b - gl["A"] @ x
        bc_ref = gl["R"] @ r_ref
        r, bc = c.residual_restrict(l, own_parts(lev, b), own_parts(lev, x))
        assert rel_err(r, own_parts(lev, r_ref)) <= TOL_KERNEL
        assert rel_err(bc, own_parts(nxt, bc_ref)) <= 4 * TOL_KERNEL
        x_ref = x + gl["P"] @ ec
        got = c.prolong_correct(l, own_parts(nxt, ec), own_parts(lev, x))
        assert rel_err(got, own_parts(lev, x_ref)) <= TOL_KERNEL


@pytest.mark.parametrize("dims,pp", PROBLEMS[:3])
def test_dot_consistent_assemble(dims, pp):
    A, h, c = make(dims, pp)
    for l, lev in enumerate(h["levels"]):
        n = h["global"]["levels"][l]["A"].shape[0]
        u, v = det_vector(n, 51), det_vector(n, 52)
        assert abs(c.dot(l, own_parts(lev, u), own_parts(lev, v)) - float(u @ v)) <= 1e-13 * np.abs(u * v).sum()
        # consistent!: ghosts <- owners, bit-exact copies
        loc = [np.concatenate([u[d["own_to_global"]], np.full(len(d["ghost_to_global"]), np.nan)]) for d in lev["parts"]]
        c.consistent(l, loc)
        for d, a in zip(lev["parts"], loc):
            assert np.array_equal(a[len(d["own_to_global"]):], u[d["ghost_to_global"]])
        # assemble!: owners += ghost copies, ghosts <- 0 (same order as the oracle => bit-exact)
        ws = [det_vector(len(d["own_to_global"]) + len(d["ghost_to_global"]), 60 + p) for p, d in enumerate(lev["parts"])]
        ref = O.assemble(lev, [w.copy() for w in ws])
        c.assemble(l, ws)
        for a, b_ in zip(ws, ref):
            assert np.allclose(a, b_, rtol=0, atol=1e-15 * 8)


@pytest.mark.parametrize("dims,pp", PROBLEMS)
@pytest.mark.parametrize("oopts", [{}, {"nu_pre": 2, "nu_post": 2}, {"smoother": "l1jacobi"},
                                   {"smoother": "chebyshev", "cheb_degree": 3}, {"nu_pre": 0, "nu_post": 2}],
                         ids=["jacobi11", "jacobi22", "l1", "cheb3", "post-only"])
def test_vcycle_parity(dims, pp, oopts):
    A, h, c = make(dims, pp, oopts)
    lev = h["levels"][0]
    n = A.shape[0]
    for seed in (71, 72):
        b = det_vector(n, seed)
        ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
        got = c.vcycle(own_parts(lev, b))
        assert rel_err(got, ref) <= TOL_VCYCLE


@pytest.mark.parametrize("dims,pp", PROBLEMS)
@pytest.mark.parametrize("oopts", [{}, {"smoother": "chebyshev", "cheb_degree": 2}], ids=["jacobi", "cheb2"])
def test_pcg_iteration_count_and_history(dims, pp, oopts):
    A, h, c = make(dims, pp, oopts)
    lev = h["levels"][0]
    n = A.shape[0]
    for b in (A @ np.ones(n) + det_vector(n, 81), det_vector(n, 82)):
        xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, b))
        x, it, hist, ok = c.pcg(own_parts(lev, b), rtol=1e-8, maxiter=200)
        assert ok and it == it_ref
        assert np.allclose(hist, hist_ref, rtol=1e-7)
        assert rel_err(x, own_of(lev, xs)) <= 1e-10
        xg = np.zeros(n)
        for d, xp in zip(lev["parts"], x):
            xg[d["own_to_global"]] = xp
        assert np.linalg.norm(b - A @ xg) <= 1.0001e-8 * np.linalg.norm(b)


@pytest.mark.parametrize("dims,pp", PROBLEMS[1:])
@pytest.mark.parametrize("tail_rows", [0, 600, 1 << 20])
def test_coarse_agglomeration_thresholds(dims, pp, tail_rows):
    """Coarse-level agglomeration (levels merged over all parts and run replicated, pamg_options.tail_rows)
    is an execution layout, not a different hierarchy: whatever the threshold, the V-cycle matches the
    oracle's N-part V-cycle to 1e-12 and PCG takes the same number of iterations.  The tail runs one launch per
    operation."""
    A, h, c = make(dims, pp, None, tail_rows=tail_rows)
    L_ = len(h["levels"])
    sizes = [h["global"]["levels"][l]["A"].shape[0] for l in range(L_)]
    want = L_ - 1 if tail_rows == 0 else next((l for l in range(1, L_) if sizes[l] <= tail_rows), L_ - 1)
    assert c.stats().tail_level == want
    lev = h["levels"][0]
    b = det_vector(A.shape[0], 77)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, b))
    x, it, hist, ok = c.pcg(own_parts(lev, b))
    assert ok and it == it_ref and np.allclose(hist, hist_ref, rtol=1e-7)


@pytest.mark.parametrize("dims,pp", [((8, 7, 6), (2, 1, 1)), ((10, 9, 8), (2, 2, 1)), ((7, 6, 6), (1, 1, 1))])
@pytest.mark.parametrize("fmt", ["auto", "sell2"])
def test_elasticity_rigid_body_sa_parity(dims, pp, fmt):
    """BASELINE config 4 at test size: 3-DOF Q1 elasticity with rigid-body near-nullspace SA (27-point node
    stencil, ~80 nnz/row, 6-DOF coarse nodes).  Device V-cycle and PCG vs the oracle on the oracle-built hierarchy."""
    nparts = int(np.prod(pp))
    A, coords = O.elasticity_q1(dims)
    B = O.rigid_body_modes(coords)
    owner = np.repeat(O.uniform_partition(pp, dims), 3).astype(np.int32)
    h = O.build(A, owner, nparts, dict(block_size=3, nullspace=B, coarse_size=60))
    c = product_context_from_oracle(h, None, **({} if fmt == "auto" else FORMATS[fmt]))
    c.device_init()
    lev = h["levels"][0]
    n = A.shape[0]
    for l, levl in enumerate(h["levels"]):
        Al = h["global"]["levels"][l]["A"]
        x = det_vector(Al.shape[0], 5 + l)
        assert rel_err(c.spmv(l, own_parts(levl, x)), own_parts(levl, Al @ x)) <= TOL_KERNEL
    b = det_vector(n, 33)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE
    rhs = A @ det_vector(n, 34)
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, rhs))
    x, it, hist, ok = c.pcg(own_parts(lev, rhs))
    assert ok and it == it_ref and np.allclose(hist, hist_ref, rtol=1e-7)
    assert rel_err(x, own_of(lev, xs)) <= 1e-9


@pytest.mark.parametrize("pp", [(2, 2, 2), (1, 1, 1)])
def test_jump_coefficient_anisotropic_diffusion_parity(pp):
    """BASELINE config 5 at test size: -div(K grad u), K = diag(k, k, 1e-3 k), k in {1, 1e4} on a checkerboard;
    strength threshold eps = 0.0831 (weak couplings filtered and lumped).  V-cycle and PCG vs the oracle, with the
    coarse levels agglomerated (replicated tail) on the multi-part layout."""
    dims = (16, 16, 16)
    nparts = int(np.prod(pp))
    A = O.diffusion_fv(dims, O.jump_coefficient_k(dims, blocks=4, kmax=1e4, eps_z=1e-3))
    owner = O.uniform_partition(pp, dims)
    oopts = {"eps_strength": 0.0831}
    h = O.build(A, owner, nparts, oopts)
    c = product_context_from_oracle(h, oopts)
    c.device_init()
    lev = h["levels"][0]
    n = A.shape[0]
    b = det_vector(n, 61)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE
    rhs = A @ det_vector(n, 62)
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, rhs), maxiter=400)
    x, it, hist, ok = c.pcg(own_parts(lev, rhs), maxiter=400)
    assert ok and it == it_ref and np.allclose(hist, hist_ref, rtol=1e-6)


def test_elasticity_product_setup_and_solve():
    """Product path end to end (gallery -> host rigid-body SA -> device PCG) at 24^3 nodes (41k DOFs)."""
    dims = (24, 24, 24)
    c = L.Context(2)
    c.gallery_elasticity(dims, (2, 1, 1))
    c.setup()
    c.device_init()
    n, nnz = c.global_size()
    b = c.host_matvec_global(det_vector(n, 3))
    own = [c.index_maps(0, p)[0] for p in range(2)]
    x, it, hist, ok = c.pcg([b[o] for o in own], rtol=1e-8, maxiter=200)
    assert ok and it < 60
    xg = np.zeros(n)
    for o, xp in zip(own, x):
        xg[o] = xp
    assert np.linalg.norm(c.host_matvec_global(xg) - b) <= 1.001e-8 * np.linalg.norm(b)


def test_pcg_graph_and_eager_agree_bitwise():
    A, h, c1 = make((20, 20, 20), (2, 2, 2), None, use_graph=1)
    _, _, c0 = make((20, 20, 20), (2, 2, 2), None, use_graph=0)
    lev = h["levels"][0]
    b = det_vector(A.shape[0], 91)
    x1, it1, h1, _ = c1.pcg(own_parts(lev, b))
    x0, it0, h0, _ = c0.pcg(own_parts(lev, b))
    assert it1 == it0 and np.array_equal(h1, h0)
    assert all(np.array_equal(a, b_) for a, b_ in zip(x1, x0))
    # a second solve on the same context replays the same graph and reproduces the same bits
    x2, it2, h2, _ = c1.pcg(own_parts(lev, b))
    assert it2 == it1 and all(np.array_equal(a, b_) for a, b_ in zip(x1, x2))
    assert c1.stats().kernel_launches > 0


def test_pcg_edge_cases():
    A, h, c = make((20, 20, 20), (1, 1, 1))
    lev = h["levels"][0]
    n = A.shape[0]
    x, it, hist, ok = c.pcg([np.zeros(n)])                     # zero rhs: 0 iterations, x = 0
    assert ok and it == 0 and np.all(x[0] == 0.0)
    x, it, hist, ok = c.pcg([det_vector(n, 5)], maxiter=0)     # no iteration allowed: x = 0, only ||r0|| recorded
    assert (not ok) and it == 0 and len(hist) == 1 and np.all(x[0] == 0.0)
    x, it, hist, ok = c.pcg([det_vector(n, 5)], maxiter=1)
    assert (not ok) and it == 1 and len(hist) == 2
    x, it, hist, ok = c.pcg([det_vector(n, 5)], maxiter=3)     # maxiter hit: reported, not raised
    assert (not ok) and it == 3 and len(hist) == 4
    xs, it_ref, _ = O.pcg(h, O.pvector_from_global(lev, det_vector(n, 5)), precond=False, maxiter=500)
    x, it, hist, ok = c.pcg([det_vector(n, 5)], precond=False, maxiter=500)   # plain CG path
    assert ok and it == it_ref


def test_part_without_rows_on_device():
    """A part that owns nothing takes part in every exchange and all-reduce with empty arrays."""
    A = O.poisson_fd((12, 12, 12))
    n = A.shape[0]
    owner = np.zeros(n, np.int32)
    owner[n // 2:] = 2
    h = O.build(A, owner, 3)
    c = product_context_from_oracle(h)
    c.device_init()
    lev = h["levels"][0]
    b = det_vector(n, 13)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, b))
    x, it, hist, ok = c.pcg(own_parts(lev, b))
    assert ok and it == it_ref and len(x[1]) == 0


def test_single_level_hierarchy_is_a_direct_solve():
    A, h, c = make((7, 5), (1, 1))
    b = det_vector(35, 7)
    x, it, hist, ok = c.pcg([b])
    assert ok and it <= 2
    assert np.linalg.norm(A @ x[0] - b) <= 1e-8 * np.linalg.norm(b)


def test_product_setup_solves_config2_shape_and_is_symmetric_preconditioner():
    """Product host setup + device solve at a size the oracle does not need to touch:
    size-independent properties (true residual, symmetry of the V-cycle operator, linearity)."""
    dims = (64, 64, 64)
    c = L.Context(1)
    c.gallery_poisson(dims, (1, 1, 1))
    c.setup()
    c.device_init()
    n = 64 ** 3
    b = c.host_matvec_global(np.ones(n))
    x, it, hist, ok = c.pcg([b])
    assert ok and hist[-1] <= 1e-8 * hist[0]
    assert np.linalg.norm(c.host_matvec_global(x[0]) - b) <= 1.001e-8 * np.linalg.norm(b)
    assert np.abs(x[0] - 1.0).max() <= 1e-6
    u, v = det_vector(n, 1), det_vector(n, 2)
    Mu, Mv = c.vcycle([u])[0], c.vcycle([v])[0]
    assert abs(v @ Mu - u @ Mv) <= 1e-10 * abs(v @ Mu)          # M symmetric (nu_pre == nu_post)
    Muv = c.vcycle([2.0 * u - 3.0 * v])[0]
    assert np.linalg.norm(Muv - (2.0 * Mu - 3.0 * Mv)) <= 1e-12 * np.linalg.norm(Muv)   # linear


@pytest.mark.parametrize("dims,pp", PROBLEMS)
@pytest.mark.parametrize("oopts", [{"cycle": "w", "coarse_size": 40}, {"cycle": "w", "coarse_size": 40, "nu_pre": 2, "nu_post": 1},
                                   {"cycle": "w", "coarse_size": 40, "smoother": "chebyshev", "cheb_degree": 2}],
                         ids=["w-jacobi11", "w-jacobi21", "w-cheb2"])
def test_w_cycle_parity(dims, pp, oopts):
    """W-cycle (pamg_options.cycle = PAMG_CYCLE_W): every coarse problem but the coarsest is visited twice, the second
    visit continuing from the first one's result.  coarse_size 40 gives 4+ levels, so the recursion really nests."""
    A, h, c = make(dims, pp, oopts)
    assert len(h["levels"]) >= 3
    lev = h["levels"][0]
    n = A.shape[0]
    b = det_vector(n, 73)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE
    hv = dict(h)
    hv["opts"] = dict(h["opts"], cycle="v")
    assert rel_err(own_of(lev, O.vcycle(hv, O.pvector_from_global(lev, b))), ref) > 1e-6   # it is not a V-cycle in disguise
    rhs = A @ det_vector(n, 74)
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, rhs))
    x, it, hist, ok = c.pcg(own_parts(lev, rhs))
    assert ok and it == it_ref and np.allclose(hist, hist_ref, rtol=1e-7)


@pytest.mark.parametrize("tail_rows", [0, 600, 1 << 20])
def test_w_cycle_with_agglomerated_tail(tail_rows):
    oopts = {"cycle": "w", "coarse_size": 40}
    A, h, c = make((20, 20, 20), (2, 2, 2), oopts, tail_rows=tail_rows)
    lev = h["levels"][0]
    b = det_vector(A.shape[0], 75)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE


@pytest.mark.parametrize("dims,pp", PROBLEMS)
@pytest.mark.parametrize("oopts", [{}, {"cycle": "w", "coarse_size": 40}], ids=["v", "w"])
def test_flexible_cg_parity(dims, pp, oopts):
    """pamg_fcg: flexible (Polak-Ribiere) AMG-preconditioned CG against the oracle's pcg(flexible=True)."""
    A, h, c = make(dims, pp, oopts)
    lev = h["levels"][0]
    n = A.shape[0]
    rhs = A @ det_vector(n, 83)
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, rhs), flexible=True)
    for rep in range(2):
        x, it, hist, ok = c.fcg(own_parts(lev, rhs))
        assert ok and it == it_ref
        assert np.allclose(hist, hist_ref, rtol=1e-7)
        assert rel_err(x, own_of(lev, xs)) <= 1e-10
    x2, it2, hist2, ok2 = c.pcg(own_parts(lev, rhs))     # switching drivers on one context re-captures the iteration graph
    xs2, it_ref2, hist_ref2 = O.pcg(h, O.pvector_from_global(lev, rhs))
    assert ok2 and it2 == it_ref2 and np.allclose(hist2, hist_ref2, rtol=1e-7)


@pytest.mark.parametrize("dims,pp", PROBLEMS)
@pytest.mark.parametrize("oopts", [{}, {"cycle": "w", "coarse_size": 40}], ids=["v", "w"])
def test_fgmres_parity(dims, pp, oopts):
    """pamg_fgmres: restarted flexible GMRES right-preconditioned by one cycle against the oracle's fgmres -- identical inner
    iteration counts, residual estimates to 1e-7, solutions; with a restart that is taken, without preconditioner, truncated."""
    A, h, c = make(dims, pp, oopts)
    lev = h["levels"][0]
    n = A.shape[0]
    rhs = A @ det_vector(n, 83)
    for kw in ({}, {"restart": 4}, {"precond": False, "restart": 12, "maxiter": 60}, {"maxiter": 3}, {"maxiter": 0}):
        xs, it_ref, hist_ref = O.fgmres(h, O.pvector_from_global(lev, rhs), **kw)
        x, it, hist, ok = c.fgmres(own_parts(lev, rhs), **kw)
        assert it == it_ref, kw
        assert ok == (hist_ref[-1] <= 1e-8 * hist_ref[0]), kw
        assert np.allclose(hist, hist_ref, rtol=1e-7), kw
        assert rel_err(x, own_of(lev, xs)) <= 1e-9, kw
    x2, it2, hist2, ok2 = c.pcg(own_parts(lev, rhs))     # the Krylov drivers share one context
    xs2, it_ref2, hist_ref2 = O.pcg(h, O.pvector_from_global(lev, rhs))
    assert ok2 and it2 == it_ref2 and np.allclose(hist2, hist_ref2, rtol=1e-7)


def test_fgmres_nonsymmetric_operator():
    """What GMRES is for: a non-symmetric operator (convection added to the 2-D Poisson values, same pattern), hierarchy built
    by the oracle from the symmetric part's pattern; CG is not applicable, FGMRES must match the oracle step for step."""
    import scipy.sparse as sp
    dims, pp = (40, 40), (2, 2)
    A0 = O.poisson_fd(dims).tocsr()
    A = A0.copy()
    rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    A.data = A.data + 0.3 * np.sign(A.indices - rows) * (np.abs(A.indices - rows) == 1)   # upwind-ish skew part along x
    owner = O.uniform_partition(pp, dims)
    h = O.build(sp.csr_matrix(A), owner, int(np.prod(pp)), {})
    c = product_context_from_oracle(h, None)
    c.device_init()
    lev = h["levels"][0]
    rhs = A @ det_vector(A.shape[0], 9)
    xs, it_ref, hist_ref = O.fgmres(h, O.pvector_from_global(lev, rhs), restart=20)
    x, it, hist, ok = c.fgmres(own_parts(lev, rhs), restart=20)
    assert ok and it == it_ref and np.allclose(hist, hist_ref, rtol=1e-7)
    assert rel_err(x, own_of(lev, xs)) <= 1e-9
    xg = np.zeros(A.shape[0])
    for d, v in zip(lev["parts"], x):
        xg[d["own_to_global"]] = v
    assert np.linalg.norm(rhs - A @ xg) <= 1.001e-8 * np.linalg.norm(rhs)


# ---- value-indexed SELL storage (kernels.cuh k_spmv_sell_vi4, k_spmv_sell_vi) -----------------------------------------------------
@pytest.mark.parametrize("dims,pp", [((28, 28, 28), (1, 1, 1)), ((33, 31, 17), (3, 2, 1)), ((200, 200), (2, 2))])
@pytest.mark.parametrize("fmt", ["sell2", "sell2-sorted"])
def test_value_indexed_sell_is_bit_identical_to_fp64_values(dims, pp, fmt, monkeypatch):
    """An operator with <= 255 distinct values is stored as columns + one byte per entry; every kernel mode must give the SAME BITS as
    the fp64-valued SELL kernels (same products, same order): all level operators, smoothers, the cycle, the PCG history.  Unsorted
    rows run four rows per lane (sell-vi), sorted rows two rows per lane (sell-vi2)."""
    monkeypatch.setenv("PAMG_VALUE_INDEX", "1")
    A, h, c = make(dims, pp, None, **FORMATS[fmt])
    assert c.stats().value_indexed[0] == 7, "level 0 of Poisson (2 / 9 / 9 distinct values in A / P / R) must be value-indexed"
    monkeypatch.setenv("PAMG_VALUE_INDEX", "0")
    A, h, c0 = make(dims, pp, None, **FORMATS[fmt])
    assert not any(c0.stats().value_indexed)
    for l in range(len(h["levels"]) - 1):
        lev, nxt = h["levels"][l], h["levels"][l + 1]
        n, nc = h["global"]["levels"][l]["A"].shape[0], h["global"]["levels"][l + 1]["A"].shape[0]
        b_, x_, ec = det_vector(n, 41), det_vector(n, 42), det_vector(nc, 43)
        for a, b in zip(c.spmv(l, own_parts(lev, x_)), c0.spmv(l, own_parts(lev, x_))):
            assert np.array_equal(a, b)
        ra, rb = c.residual_restrict(l, own_parts(lev, b_), own_parts(lev, x_)), c0.residual_restrict(l, own_parts(lev, b_), own_parts(lev, x_))
        for a, b in zip(ra[0] + ra[1], rb[0] + rb[1]):
            assert np.array_equal(a, b)
        for a, b in zip(c.prolong_correct(l, own_parts(nxt, ec), own_parts(lev, x_)), c0.prolong_correct(l, own_parts(nxt, ec), own_parts(lev, x_))):
            assert np.array_equal(a, b)
        for a, b in zip(c.smooth(l, 2, own_parts(lev, b_), own_parts(lev, x_)), c0.smooth(l, 2, own_parts(lev, b_), own_parts(lev, x_))):
            assert np.array_equal(a, b)
    lev = h["levels"][0]
    rhs = A @ det_vector(A.shape[0], 17)
    for a, b in zip(c.vcycle(own_parts(lev, rhs)), c0.vcycle(own_parts(lev, rhs))):
        assert np.array_equal(a, b)
    (x, it, hist, ok), (x0, it0, hist0, ok0) = c.pcg(own_parts(lev, rhs)), c0.pcg(own_parts(lev, rhs))
    assert ok and ok0 and it == it0
    families = {t[0] for t in map(str.split, c.trace_names()) if len(t) >= 3 and t[2] == "A0"}
    assert families == {"sell-vi" if fmt == "sell2" else "sell-vi2"}, families
    if fmt == "sell2":
        # four rows per lane: the FUSED DOT PRODUCTS add their per-thread partials in another order (another row -> thread map), so
        # the PCG scalars differ in the last bits; every operator result above is still bit-identical
        assert np.allclose(hist, hist0, rtol=1e-11) and rel_err(x, x0) <= 1e-11
    else:
        assert np.array_equal(hist, hist0)
        for a, b in zip(x, x0):
            assert np.array_equal(a, b)
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, rhs))           # and the oracle, as for every other format
    assert it == it_ref and np.allclose(hist, hist_ref, rtol=1e-7)


@pytest.mark.parametrize("smoother", ["l1jacobi", "chebyshev"])
def test_value_indexed_sell_other_smoothers(smoother, monkeypatch):
    monkeypatch.setenv("PAMG_VALUE_INDEX", "1")
    oopts = {"smoother": smoother}
    A, h, c = make((20, 20, 20), (2, 2, 2), oopts, **FORMATS["sell2"])
    assert c.stats().value_indexed[0] == 7
    lev = h["levels"][0]
    b = det_vector(A.shape[0], 5)
    ref = own_of(lev, O.vcycle(h, O.pvector_from_global(lev, b)))
    assert rel_err(c.vcycle(own_parts(lev, b)), ref) <= TOL_VCYCLE
    xs, it_ref, hist_ref = O.pcg(h, O.pvector_from_global(lev, b))
    x, it, hist, ok = c.pcg(own_parts(lev, b))
    assert ok and it == it_ref and np.allclose(hist, hist_ref, rtol=1e-7)
