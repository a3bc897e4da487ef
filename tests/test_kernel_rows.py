"""Every SpMV kernel family, row by row, against a sequential and an extended-precision reference.

The other GPU tests take their operators from the gallery (Poisson, jump coefficients, elasticity) and compare norm-wise.  Here
synthetic operators are uploaded as a two-level hierarchy (A, P, R = P^T, coarse A_c = R A P solved by its inverse) so that each
kernel family meets the shapes where kernels go wrong: n in {1, 31, 127, 128, 129, 4097}, 1-entry rows and empty rows, rows at
the CSR-stream cap, uneven rows inside one slice, dictionaries at their size limits (-0.0 among the values, exponents over
+-150), 1 to 32 diagonals with offsets up to n/2, boundary rows of uneven parts, and launches that stride over the slices more
than once.  Every case asserts the kernel it reached (pamg_stats, and the launch names of one PCG iteration), so a change of
dispatch cannot turn it into a test of something else.

Two references, both checked ROW BY ROW:
  (a) the fp64 sequential sum s = s + a_ij * x_j in stored column order, each product rounded before the add.  The CSR-stream
      (short rows), SELL, value-indexed SELL (both index widths) and implied-column SELL kernels must match it bit for bit on
      every row without own-ghost entries (np.array_equal), in the MUL, RESID (b - s), ADD (x + s) and RESTRICT epilogues;
  (b) the same sum in np.longdouble (64-bit significand).  Everything else -- the sub-warp CSR kernels (strided lanes, tree
      reduction), CSR-stream with long rows (16 lanes per row), boundary rows (own part, then ghost part), the smoother
      epilogues (nvcc may contract x + w (b - s) into an FMA) and the fused dot products -- must lie within a componentwise
      bound derived from the operation, with gamma_k = k u / (1 - k u), u = 2^-53.  The bounds add the error of reference (b)
      itself (gamma with u = 2^-64).
"""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp

import amg_oracle as O
from parallel_amg_b200 import _lib as L
from util import det_vector, own_parts, product_context_from_oracle

LD = np.longdouble
HAVE_LD = np.finfo(LD).nmant >= 63
U = 2.0 ** -53
U_LD = 2.0 ** -64
RED_GRID = 148 * 8     # kernels.cuh: upper bound of the CTAs of a bounded (one resident wave) launch
SLICE_ROWS = 128       # rows per slice of the four-rows-per-lane value-indexed and implied-column layouts
EXACT = {"stream", "sell", "sell-vi", "sell-vi2", "sell-vi16", "sell-diag"}   # row sums in stored column order
FAMILIES = ("sell-diag", "sell-vi16", "sell-vi2", "sell-vi", "sell", "stream-long", "stream", "csr")
FORMAT_OF = {"csr": L.FORMAT_CSR, "stream": L.FORMAT_STREAM, "stream-long": L.FORMAT_STREAM}

need_ld = pytest.mark.skipif(not HAVE_LD, reason="reference (b) needs a long double with a 64-bit significand")


def gamma(k, u=U):
    k = np.asarray(k, dtype=LD)
    return k * LD(u) / (LD(1) - k * LD(u))


def gamma2(k):
    """gamma_k plus the error of reference (b), which is computed with gamma_k at u = 2^-64"""
    return gamma(k) + gamma(k, U_LD)


# ---- operators ---------------------------------------------------------------------------------------------------------------
def _csr(rows, cols, vals, shape):
    M = sp.csr_matrix((np.asarray(vals, np.float64), (np.asarray(rows, np.int64), np.asarray(cols, np.int64))), shape=shape)
    M.sort_indices()   # coo -> csr keeps explicit (signed) zeros; there are no duplicates to sum
    return M


def irregular(n, seed=1, maxdeg=12, long_rows=None, vals=None, diag=None):
    """Symmetric, random partners (0 .. 2 maxdeg per row); rows 3, 10, 17, ... hold only their diagonal; long_rows {row: length}
    get exactly that many entries.  vals: off-diagonal values, round robin over the pairs (all of them used once there are
    enough pairs); None: -(0.25 .. 1.25), ~1000 distinct.  diag: the diagonal value; None: the row's absolute off-diagonal sum
    times 1 + 2^-20 (1 for a lone diagonal), diagonally dominant by a hair: with x close to a constant vector every row sum
    cancels (sum |a_ij x_j| ~ 1e6 |sum a_ij x_j|)."""
    rng = np.random.default_rng(seed)
    long_rows = long_rows or {}
    quiet = np.zeros(n, bool)
    quiet[3::7] = True
    for i in long_rows:
        quiet[i] = True
    deg = rng.integers(0, maxdeg + 1, n)
    deg[quiet] = 0
    r = np.repeat(np.arange(n), deg)
    c = rng.integers(0, n, r.size)
    keep = (r != c) & ~quiet[c]
    r, c = r[keep], c[keep]
    free = np.flatnonzero(~quiet)
    for i, m in long_rows.items():
        r = np.concatenate([r, np.full(m - 1, i)])
        c = np.concatenate([c, rng.choice(free, m - 1, replace=False)])
    key = np.unique(np.minimum(r, c) * n + np.maximum(r, c))
    lo, hi = key // n, key % n
    if vals is None:
        v = -(0.25 + ((lo * 7 + hi * 13) % 1000) / 1000.0)
    else:
        v = np.asarray(vals, np.float64)[np.arange(len(lo)) % len(vals)]
    absum = np.bincount(lo, np.abs(v), n) + np.bincount(hi, np.abs(v), n)
    d = absum * (1.0 + 2.0 ** -20) + (absum == 0) if diag is None else np.full(n, float(diag))
    i = np.arange(n)
    return _csr(np.concatenate([lo, hi, i]), np.concatenate([hi, lo, i]), np.concatenate([v, v, d]), (n, n))


def stencil(n, offs, nvals, diag=40.0):
    """Entries at row + o for every o in offs (0 <= row + o < n).  Off the diagonal, the pairs {i, j} take the nvals - 1 values
    in [-1, -0.5) round robin (symmetric when offs is; all used once there are enough pairs); the diagonal is `diag`: at most
    nvals distinct values.  |vals| <= 1 and diag 40 > 2 * 31: the symmetric part is diagonally
    dominant for up to 32 offsets."""
    i = np.arange(n)
    rows, cols = [], []
    for o in sorted(set(offs)):
        ok = (i + o >= 0) & (i + o < n)
        rows.append(i[ok])
        cols.append(i[ok] + o)
    r, c = np.concatenate(rows), np.concatenate(cols)
    m = max(nvals - 1, 1)
    vals = -(0.5 + 0.5 * np.arange(m) / m)
    off = r != c
    pair = np.unique(np.minimum(r, c)[off] * n + np.abs(r - c)[off], return_inverse=True)[1].ravel()   # (i, j) and (j, i): one pair
    v = np.full(len(r), float(diag))
    v[off] = vals[pair % m]
    assert nvals > 1 or np.all(r == c)
    return _csr(r, c, v, (n, n))


def wide_values(k):
    """k distinct values: -0.0 and +-(1 + j / 2k) 2^e with the exponents e spread over [-150, 150]"""
    j = np.arange(k - 1)
    e = j * 301 // max(k - 1, 1) - 150
    v = np.where(j % 2 == 0, -1.0, 1.0) * np.ldexp(1.0 + j / (2.0 * k), e)
    return np.concatenate([[-0.0], v])


def prolongator(A, owner, nc):
    """Aggregation-like P (n x ~nc) and the owners of its columns.  Each part's rows, in order, form aggregates of at least two
    rows, owned by the part; row i -> its aggregate (value 1) except every fifth row of a part, which stays empty; every third
    row also 0.25 on the aggregate of its first off-diagonal neighbour in A, so that, as for a smoothed prolongator, P and
    R = P^T only couple A-neighbours.  Every aggregate keeps a non-empty row: P has full column rank, A_c = P^T A P is
    invertible."""
    n = A.shape[0]
    agg, pos, cown = np.zeros(n, np.int64), np.zeros(n, np.int64), []
    for p in range(int(owner.max()) + 1):
        rows = np.flatnonzero(owner == p)
        if len(rows) == 0:
            continue
        ncp = max(1, min(round(nc * len(rows) / n), len(rows) // 2))
        pos[rows] = np.arange(len(rows))
        agg[rows] = len(cown) + pos[rows] * ncp // len(rows)
        cown += [p] * ncp
    i = np.arange(n)
    has = pos % 5 != 4
    lens = np.diff(A.indptr)
    first = np.where(A.indices[A.indptr[:-1]] != i, A.indices[A.indptr[:-1]], A.indices[np.minimum(A.indptr[:-1] + 1, A.nnz - 1)])
    two = has & (pos % 3 == 0) & (lens > 1) & (agg[first] != agg)
    P = _csr(np.concatenate([i[has], i[two]]), np.concatenate([agg[has], agg[first[two]]]),
             np.concatenate([np.ones(has.sum()), np.full(two.sum(), 0.25)]), (n, len(cown)))
    return P, np.asarray(cown, np.int32)


def three_parts(A):
    """60 % / ~40 % / six rows: the six rows of part 2 all have partners in the other parts (every row a boundary row)"""
    n = A.shape[0]
    owner = np.zeros(n, np.int32)
    owner[int(0.6 * n):] = 1
    owner[np.flatnonzero(np.diff(A.indptr) > 3)[-6:]] = 2
    return owner


def hierarchy(A, P, owner, cown, nparts, oopts=None):
    """Two-level hierarchy of the oracle's localised form: level 0 (A, P, R = P^T), level 1 A_c = R A P with inv(A_c)."""
    n, nc = P.shape
    R = P.T.tocsr()
    R.sort_indices()
    Ac = O.spgemm_structural(R, O.spgemm_structural(A, P))
    gh = dict(levels=[dict(A=A, owner=np.asarray(owner, np.int32), P=P, R=R, agg_local=np.zeros(n, np.int32)), dict(A=Ac, owner=cown)],
              coarse_inv=np.linalg.inv(Ac.toarray()), opts=O.options(**(oopts or {})), nparts=nparts)
    h = O.localize(gh)
    h["rho_dinv_a"] = [O.estimate_rho(lev["A"], 1.0 / lev["A"].diagonal()) for lev in gh["levels"]]
    h["global"] = gh
    return h


# ---- the cases: (name, n) -> operator, options, the kernel family it exists for -----------------------------------------------
ALL_N = (1, 31, 127, 128, 129, 4097)
STREAM_LONG_ROWS = {1000: 3069, 1001: 3069, 1002: 3069, 1003: 3069}   # the cap; consecutive, so their first entries cover all residues mod 4
CASE_SHAPES = {
    **{f"csr-lanes{ln}": ALL_N for ln in (1, 2, 4, 8, 16, 32)},
    "csr-fallback": (4097,),
    "stream": ALL_N,
    "stream-long": (129, 4097),
    **{f"sell{r}-sigma{s}": ALL_N for r in (1, 2) for s in (1, 256)},
    "sell-vi2-sorted": (128, 129, 4097),
    "vi4-255": ALL_N, "vi4-256": (128, 129, 4097), "vi4-4095": (4097,), "vi4-4096": (4097,),
    "diag-1-1": ALL_N, "diag-2-2": ALL_N, "diag-7-254": ALL_N, "diag-31-2": (127, 128, 129, 4097), "diag-32-254": (127, 128, 129, 4097),
    "diag-7-255": (129, 4097),
    **{f"boundary-fuse{f}": (129, 4097) for f in (0, 1)},
}
GRID = [(c, n) for c, shapes in CASE_SHAPES.items() for n in shapes]


def diag_offsets(nd, n):
    if nd == 1:
        return [0]
    if nd == 2:
        return [0, 1]
    if nd == 7:
        return [-(n // 2), -2, -1, 0, 1, 2, n // 2]
    if nd == 31:
        return list(range(-15, 16))
    return list(range(-15, 16)) + [n // 2]


@functools.lru_cache(maxsize=4)
def case(name, n):
    """dict(h, opts, env, want {(op, mode): family}, ndist / ndiag expectations)"""
    s = dict(opts={}, env={}, want={}, nparts=1, ndist=None, ndiag=None)
    nc = n // 8
    if name.startswith("csr-lanes"):
        A = irregular(n)
        s["opts"] = dict(spmv_format=L.FORMAT_CSR, lanes_per_row=int(name[9:]))
        s["want"] = {("A0", "resid"): "csr"}
    elif name == "csr-fallback":
        A = irregular(n, long_rows={1000: 3070})
        s["opts"] = dict(spmv_format=L.FORMAT_STREAM)
        s["want"] = {("A0", "resid"): "csr"}
    elif name == "stream":
        A = irregular(n, long_rows=STREAM_LONG_ROWS if n > 4000 else None)
        s["opts"] = dict(spmv_format=L.FORMAT_STREAM)
        s["want"] = {("A0", "resid"): "stream", ("R0", "restrict"): "stream"}
    elif name == "stream-long":
        A = irregular(n)
        nc = n // 64                                                             # R rows: ~70 entries (mean >= 48)
        s["opts"] = dict(spmv_format=L.FORMAT_STREAM)
        s["want"] = {("A0", "resid"): "stream", ("R0", "restrict"): "stream-long"}
    elif name.startswith("sell") and "sigma" in name:
        A = irregular(n)
        s["opts"] = dict(spmv_format=L.FORMAT_SELL, sell_rows_per_thread=int(name[4]), sell_sigma=int(name.split("sigma")[1]))
        if n < 4097:                                                             # 4097 rows carry > 4095 distinct values
            s["env"] = {"PAMG_VALUE_INDEX": "0"}
        s["want"] = {("A0", "resid"): "sell"}
    elif name == "sell-vi2-sorted":
        # one row of 40 entries per 64: unsorted fill > 2, so the automatic sigma sorts, and sorted rows take the two-row kernel
        A = irregular(n, maxdeg=2, long_rows={i: 40 for i in range(5, n, 64)}, vals=-(0.5 + np.arange(20) / 40.0), diag=64.0)
        s["opts"] = dict(spmv_format=L.FORMAT_SELL)
        s["want"] = {("A0", "resid"): "sell-vi2"}
    elif name.startswith("vi4-"):
        k = int(name[4:])
        A = irregular(n, vals=wide_values(k - 1), diag=2.0 ** 160)             # k - 1 off-diagonal values (-0.0 among them) + 2^160
        s["opts"] = dict(spmv_format=L.FORMAT_SELL, sell_sigma=1)
        s["want"] = {("A0", "resid"): {255: "sell-vi", 256: "sell-vi16", 4095: "sell-vi16", 4096: "sell"}[k]}
        s["ndist"] = k if n >= 128 else None
    elif name.startswith("diag-"):
        nd, k = map(int, name[5:].split("-"))
        offs = diag_offsets(nd, n)
        A = stencil(n, offs, k)
        s["opts"] = dict(spmv_format=L.FORMAT_SELL_DIAG)
        s["want"] = {("A0", "resid"): "sell-vi" if k == 255 else "sell-diag"}
        s["ndist"] = k if n >= 127 else None
        s["ndiag"] = len({o for o in offs if abs(o) < n})
    elif name.startswith("boundary"):
        A = irregular(n)
        s["opts"] = dict(spmv_format=L.FORMAT_STREAM)
        s["env"] = {"PAMG_FUSE_HALO": name[-1]}
        s["nparts"] = 3
        s["want"] = {("A0", "resid"): "stream"}
    else:
        raise KeyError(name)
    owner = three_parts(A) if s["nparts"] == 3 else np.zeros(n, np.int32)
    P, cown = prolongator(A, owner, nc)
    s["h"] = hierarchy(A, P, owner, cown, s["nparts"])
    return s


def distinct_values(M):
    """distinct values by bit pattern, +0.0 not counted (the layouts' dictionary entry 0)"""
    b = np.unique(M.data.view(np.uint64))
    return int(np.count_nonzero(b))


# ---- references ----------------------------------------------------------------------------------------------------------------
def seq_rows(M, x, dtype=np.float64):
    """Row sums s = s + a_ij * x_j in stored order, vectorised over rows by entry position.  dtype float64: reference (a), each
    product rounded to fp64 before the add; longdouble: reference (b)."""
    n = M.shape[0]
    s = np.zeros(n, dtype)
    if M.nnz == 0:
        return s
    prod = M.data.astype(dtype) * np.asarray(x)[M.indices].astype(dtype)
    lens = np.diff(M.indptr)
    beg = M.indptr[:-1]
    for k in range(int(lens.max())):
        ok = np.flatnonzero(lens > k)
        s[ok] = s[ok] + prod[beg[ok] + k]
    return s


def ext_rows(pairs, n):
    """Reference (b) over one or more blocks of the same rows: (sum a_ij x_j, sum |a_ij x_j|, entries per row)"""
    s, S, k = np.zeros(n, LD), np.zeros(n, LD), np.zeros(n, np.int64)
    for M, x in pairs:
        s += seq_rows(M, x, LD)
        S += seq_rows(abs(M), np.abs(x), LD)
        k += np.diff(M.indptr)
    return s, S, k


def assert_bits(what, rows, got, ref):
    bad = np.flatnonzero(got != ref)
    if bad.size:
        i = bad[0]
        raise AssertionError(f"{what}: {bad.size} of {len(got)} rows differ from the sequential sum; first: row {rows[i]}, got {got[i]!r}, "
                             f"reference {ref[i]!r}")


def assert_bounded(what, rows, got, ref, bound):
    assert np.all(np.isfinite(got)), f"{what}: non-finite result in row {rows[np.flatnonzero(~np.isfinite(got))[0]]}"
    err = np.abs(got.astype(LD) - ref)
    over = err > bound
    if over.any():
        i = int(np.argmax(np.where(over, err / np.maximum(bound, LD(1e-300)), -1)))
        raise AssertionError(f"{what}: {int(over.sum())} of {len(got)} rows outside the bound; worst: row {rows[i]}, got {got[i]!r}, "
                             f"reference {float(ref[i])!r}, |error| {float(err[i]):.3e} > bound {float(bound[i]):.3e}")


def gather(level, vs, n):
    g = np.zeros(n)
    for d, v in zip(level["parts"], vs):
        g[d["own_to_global"]] = v[: len(d["own_to_global"])]
    return g


def check_op(what, h, key, xin, got, fam, mode="mul", in0=None):
    """Rows of y = key x (key A: level-0 rows and columns; P: columns coarse; R: rows coarse), per part.

    mode mul / restrict: y = s; resid: y = b - s (in0 = b); add: y = x + s (in0 = x).
    Rows without own-ghost entries of an EXACT family: bit for bit equal to reference (a) with the same epilogue in fp64.
    Every other row: |y^ - y| <= gamma_{k+c} T, k = entries of the row, c = roundings of the epilogue (0 for mul, 1 for b - s and
    x + s), T = sum_j |a_ij x_j| (+ |in0_i|): the row sum of k products in any order and any association (sequential, strided
    lanes, tree reduction, own part + ghost part) is within gamma_k sum |a_ij x_j| of the exact sum, the epilogue adds one
    rounding of at most u |result|."""
    lev0, lev1 = h["levels"]
    rlev, clev = {"A": (lev0, lev0), "P": (lev0, lev1), "R": (lev1, lev0)}[key]
    for p, d in enumerate(lev0["parts"]):
        rows = rlev["parts"][p]["own_to_global"]
        cd = clev["parts"][p]
        Moo, Mog = d[key + "_oo"], d[key + "_og"]
        xo, xg = xin[cd["own_to_global"]], xin[cd["ghost_to_global"]]
        sb, S, k = ext_rows([(Moo, xo), (Mog, xg)] if Mog.shape[1] else [(Moo, xo)], len(rows))
        sa = seq_rows(Moo, xo)
        if mode in ("mul", "restrict"):
            ra, rb, T, c = sa, sb, S, 0
        else:
            e0 = in0[rows]
            sign = -1.0 if mode == "resid" else 1.0
            ra, rb, T, c = e0 + sign * sa, e0.astype(LD) + LD(sign) * sb, np.abs(e0).astype(LD) + S, 1
        y = got[p]
        exact = (np.diff(Mog.indptr) == 0) & (fam in EXACT)
        assert_bits(f"{what} [{fam}, part {p}]", rows[exact], y[exact], ra[exact])
        assert_bounded(f"{what} [{fam}, part {p}]", rows[~exact], y[~exact], rb[~exact], gamma2(k[~exact] + c) * T[~exact])


def launch_families(c):
    """{(operator, mode): family} from the launch names of the last captured PCG iteration"""
    fam = {}
    names = c.trace_names()
    for nm in names:
        t = nm.split()
        if len(t) >= 3 and t[0] in FAMILIES:
            fam[(t[2], t[1])] = t[0]
    return fam, names


def check_cg_step(what, c, h, b, precond):
    """One CG step from x0 = 0: p = z0 (= b, or the V-cycle of b), x1 = alpha p with alpha = (b . z0) / (z0 . A z0).

    x1 / z0 must be one constant to 1 ulp (x1_i = fl(alpha^ z0_i)): PCG stepped along exactly the z0 that pamg_vcycle returns.
    That constant alpha^ = rho^ / sigma^ is checked against alpha in extended precision.  The fused dot products carry
      |rho^ - rho| <= gamma_n sum |b_i z_i|,
      |sigma^ - sigma| <= gamma_n sum |z_i| (|q_i| + E_i) + sum |z_i| E_i,   E_i = gamma_{k_i} sum_j |a_ij z_j| (the row bound of q^ = A z),
    so |alpha^ / alpha - 1| <= (1 + e_rho)(1 + u) / (1 - e_sigma) - 1 =: e, with e_rho, e_sigma the relative bounds above.
    hist[1] = ||r1||, r1_i = b_i - alpha^ q^_i rounded twice (or once, contracted):
      |r1^_i - r1_i| <= |alpha| (1 + e) E_i + e |alpha| |q_i| + gamma_2 (|b_i| + |alpha| (1 + e) (|q_i| + E_i)) =: F_i,
    and the computed norm sqrt(fl(sum r1^_i^2)) is within (sqrt(1 + gamma_n)(1 + u) - 1) ||r1^|| of ||r1^||."""
    lev0 = h["levels"][0]
    A = h["global"]["levels"][0]["A"]
    n = A.shape[0]
    z = gather(lev0, c.vcycle(own_parts(lev0, b)), n) if precond else b
    x, it, hist, ok = c.pcg(own_parts(lev0, b), maxiter=1, precond=precond)
    assert it == 1 and len(hist) == 2, (what, it, hist)
    x1 = gather(lev0, x, n)
    nz = z != 0
    assert nz.any() and np.all(x1[~nz] == 0), what
    ratio = x1[nz].astype(LD) / z[nz].astype(LD)
    a_hat = np.median(ratio)
    spread = (ratio.max() - ratio.min()) / abs(a_hat)
    assert spread <= 2 * U + 2.0 ** -62, f"{what}: x1 / z0 is not one constant (relative spread {float(spread):.3e}): not a step along z0"
    bl, zl = b.astype(LD), z.astype(LD)
    q, S, k = ext_rows([(A, z)], n)
    E = gamma2(k) * S
    rho, sigma = np.sum(bl * zl), np.sum(zl * q)
    e_rho = (gamma2(n) * np.sum(np.abs(bl * zl))) / abs(rho)
    e_sig = (gamma2(n) * np.sum(np.abs(zl) * (np.abs(q) + E)) + np.sum(np.abs(zl) * E)) / abs(sigma)
    assert e_sig < 0.5, f"{what}: z . A z is not resolved in fp64 (relative bound {float(e_sig):.2e})"
    e = (1 + e_rho) * (1 + LD(U)) / (1 - e_sig) - 1
    alpha = rho / sigma
    assert abs(a_hat - alpha) <= e * abs(alpha) + 2 * U * abs(a_hat), \
        f"{what}: alpha {float(a_hat)!r}, extended {float(alpha)!r}, |error| {float(abs(a_hat - alpha)):.3e} > {float(e * abs(alpha)):.3e}"
    cn = np.sqrt(1 + gamma2(n)) * (1 + LD(U)) - 1
    nb = np.sqrt(np.sum(bl * bl))
    assert abs(LD(hist[0]) - nb) <= cn * nb, (what, hist[0], float(nb))
    aa = abs(alpha) * (1 + e)
    F = aa * E + e * abs(alpha) * np.abs(q) + gamma2(2) * (np.abs(bl) + aa * (np.abs(q) + E))
    nr, nF = np.sqrt(np.sum((bl - alpha * q) ** 2)), np.sqrt(np.sum(F * F))
    bound = nF + cn * (nr + nF)
    assert abs(LD(hist[1]) - nr) <= bound, f"{what}: ||r1|| {hist[1]!r}, extended {float(nr)!r}, bound {float(bound):.3e}"


def vi_bits_ok(fam, vi):
    return {"sell": vi & 1 == 0, "sell-vi": vi & (1 | 8 | 64) == 1, "sell-vi2": vi & (1 | 8 | 64) == 1,
            "sell-vi16": vi & (1 | 8 | 64) == 9, "sell-diag": vi & (1 | 8 | 64) == 65}.get(fam, vi & 1 == 0)


def device_context(s, monkeypatch, oopts=None, h=None):
    for k, v in s["env"].items():
        monkeypatch.setenv(k, v)
    c = product_context_from_oracle(h or s["h"], oopts, **s["opts"])
    c.device_init()
    return c


def assert_family(what, s, c, fam, names):
    famA = fam[("A0", "resid")]
    for key, want in s["want"].items():
        assert fam.get(key) == want, (what, key, fam.get(key), want, names)
    st = c.stats()
    assert st.format[0] == FORMAT_OF.get(famA, L.FORMAT_SELL), (what, famA, st.format[0])
    assert vi_bits_ok(famA, st.value_indexed[0]), (what, famA, st.value_indexed[0])
    if "lanes_per_row" in s["opts"]:
        assert st.lanes[0] == s["opts"]["lanes_per_row"], what
    if s["nparts"] > 1:
        assert "k_boundary" in names and st.fused_halo == 0, what   # all parts on one GPU: the boundary role is a launch of its own
    return famA


# ---- no GPU: every operator lands in the layout its case names; the references -------------------------------------------------
@pytest.mark.parametrize("name,n", GRID, ids=[f"{c}-n{n}" for c, n in GRID])
def test_operator_lands_in_its_layout(name, n):
    s = case(name, n)
    h = s["h"]
    c = product_context_from_oracle(h, None, **s["opts"])
    A0 = h["levels"][0]["parts"][0]["A_oo"]
    lens = np.diff(A0.indptr)
    if name.startswith("csr-lanes") and n > 3:
        assert (lens == 1).any() and (np.diff(h["global"]["levels"][0]["P"].indptr) == 0).any()   # 1-entry rows of A, empty rows of P
    elif name == "csr-fallback":
        assert lens.max() == 3070 and c.layout_stream(0, 0, L.A_OO) is None
    elif name == "stream":
        assert c.layout_stream(0, 0, L.A_OO) is not None
        if n == 4097:
            assert lens.max() == 3069 and sorted(A0.indptr[list(STREAM_LONG_ROWS)] % 4) == [0, 1, 2, 3]
        Rl = np.diff(h["levels"][0]["parts"][0]["R_oo"].indptr)
        assert Rl.mean() < 48
    elif name == "stream-long":
        assert c.layout_stream(0, 0, L.R_OO) is not None and np.diff(h["levels"][0]["parts"][0]["R_oo"].indptr).mean() >= 48
    elif name.startswith("sell") and "sigma" in name:
        if n == 4097:
            assert c.layout_sell_values(0, 0, L.A_OO, 128, -4) is None                  # > 4095 distinct values: fp64 SELL
        sl = c.layout_sell(0, 0, L.A_OO, 32 * s["opts"]["sell_rows_per_thread"], s["opts"]["sell_sigma"])
        assert np.ptp(lens) > 4 or n < 31                                                 # uneven rows
        if n > 1:
            assert sl["permuted"] == (s["opts"]["sell_sigma"] > 1)
    elif name == "sell-vi2-sorted":
        vi = c.layout_sell_values(0, 0, L.A_OO, 64, 1)
        assert vi is not None and vi[1].dtype == np.uint8
        unsorted, srt = c.layout_sell(0, 0, L.A_OO, 64, 1), c.layout_sell(0, 0, L.A_OO, 64, 64 * 64)
        fill = lambda lay: len(lay["col"]) / A0.nnz                                      # noqa: E731
        assert fill(unsorted) > 2.0 and srt["permuted"] and fill(srt) < fill(unsorted) - 0.02
    elif name.startswith("vi4-"):
        k = int(name[4:])
        if s["ndist"]:
            assert distinct_values(A0) == k
        vi = c.layout_sell_values(0, 0, L.A_OO, 128, -4)
        width = 1 if distinct_values(A0) <= 255 else 2 if distinct_values(A0) <= 4095 else None
        assert (vi is None) if width is None else (vi is not None and vi[1].dtype.itemsize == width)
        if vi is not None and n > 1:
            assert np.any(vi[0].view(np.uint64) == np.uint64(1 << 63))                   # -0.0 is a dictionary entry of its own
            assert np.abs(np.frexp(vi[0][vi[0] != 0])[1]).max() >= 140                    # exponents beyond +-140
    elif name.startswith("diag-"):
        k = int(name.split("-")[2])
        if s["ndist"]:
            assert distinct_values(A0) == k
        lay = c.layout_sell_diag(0, 0)
        if k == 255:
            assert lay is None and c.layout_sell_values(0, 0, L.A_OO, 128, -4)[1].dtype == np.uint8
        else:
            assert lay is not None and len(lay["off"]) == s["ndiag"], (lay and lay["off"], s["ndiag"])
            nd = int(name.split("-")[1])
            assert np.abs(lay["off"]).max() == max(abs(o) for o in diag_offsets(nd, n) if abs(o) < n)
    elif name.startswith("boundary"):
        own = [len(d["own_to_global"]) for d in h["levels"][0]["parts"]]
        assert len(set(own)) == 3 and own[2] == 6
        bnd = [c.layout_boundary(0, p, L.A_OO) for p in range(3)]
        assert len(bnd[2]["rows"]) == own[2]                                              # every row of part 2 is a boundary row
        assert all(0 < len(bnd[p]["rows"]) < own[p] for p in (0, 1))                      # interior and boundary rows


@need_ld
def test_sequential_reference_is_scipys_product():
    """Reference (a) is the order scipy's CSR product uses (one rounded product, one add per entry, stored order)."""
    for A in (irregular(4097, long_rows=STREAM_LONG_ROWS), stencil(4097, diag_offsets(7, 4097), 254), irregular(500, vals=wide_values(255), diag=2.0 ** 160)):
        for x in (det_vector(A.shape[0], 3), 1.0 + 2.0 ** -30 * det_vector(A.shape[0], 4)):
            assert np.array_equal(seq_rows(A, x), A @ x)


@need_ld
def test_extended_reference_agrees_with_fsum():
    """Reference (b) on sampled rows (cancelling ones included) against the exact sum: math.fsum of the exact products
    (Fraction), and within gamma_k(2^-64) sum |a_ij x_j| of it."""
    A = irregular(4097, long_rows=STREAM_LONG_ROWS)
    x = 1.0 + 2.0 ** -30 * det_vector(4097, 4)
    s, S, k = ext_rows([(A, x)], 4097)
    for i in list(range(0, 4097, 97)) + list(STREAM_LONG_ROWS):
        a, j = A.data[A.indptr[i]:A.indptr[i + 1]], A.indices[A.indptr[i]:A.indptr[i + 1]]
        exact = sum(Fraction(float(v)) * Fraction(float(x[c])) for v, c in zip(a, j))
        ref = math.fsum(float(v) * float(x[c]) for v, c in zip(a, j))      # products rounded, exact sum
        assert abs(Fraction(ref) - exact) <= Fraction(float(U)) * Fraction(float(S[i])) * 2
        assert abs(Fraction(float(s[i])) - exact) <= Fraction(float(gamma(k[i], U_LD) * S[i])) + Fraction(abs(float(s[i]))) * Fraction(float(U))
        assert S[i] > 1e5 * abs(s[i]) or k[i] < 3                                        # the rows cancel


# ---- GPU: every operator row, both dot products of one CG step ----------------------------------------------------------------
@need_ld
@pytest.mark.gpu
@pytest.mark.parametrize("name,n", GRID, ids=[f"{c}-n{n}" for c, n in GRID])
def test_kernel_rows(name, n, monkeypatch):
    s = case(name, n)
    h = s["h"]
    c = device_context(s, monkeypatch)
    nc = h["global"]["levels"][1]["A"].shape[0]
    lev0, lev1 = h["levels"]
    A = h["global"]["levels"][0]["A"]
    b = det_vector(n, 5)
    check_cg_step(f"{name} n={n} PCG", c, h, b, precond=True)
    fam, names = launch_families(c)
    famA = assert_family(name, s, c, fam, names)
    famP, famR = fam[("P0", "add")], fam[("R0", "restrict")]
    assert fam[("A0", "jacobi+dot")] == famA
    check_cg_step(f"{name} n={n} CG", c, h, b, precond=False)
    fam2, _ = launch_families(c)
    assert fam2[("A0", "mul+dot")] == famA
    for seed, xv in ((1, det_vector(n, 11)), (2, 1.0 + 2.0 ** -30 * det_vector(n, 12))):   # the second cancels where the diagonal barely dominates
        what = f"{name} n={n} x{seed}"
        check_op(f"{what} A x", h, "A", xv, c.spmv(0, own_parts(lev0, xv)), famA)
        bv = A @ xv if seed == 2 else det_vector(n, 13)                                     # b - A x cancels too
        r, bc = c.residual_restrict(0, own_parts(lev0, bv), own_parts(lev0, xv))
        check_op(f"{what} b - A x", h, "A", xv, r, famA, "resid", bv)
        check_op(f"{what} R r", h, "R", gather(lev0, r, n), bc, famR, "restrict")
        ec = det_vector(nc, 14 + seed)
        check_op(f"{what} x + P e", h, "P", ec, c.prolong_correct(0, own_parts(lev1, ec), own_parts(lev0, xv)), famP, "add", xv)
    c.close()


# ---- GPU: the smoother epilogues ------------------------------------------------------------------------------------------------
SMOOTH_GRID = [("csr-lanes8", 129), ("stream", 4097), ("sell2-sigma1", 129), ("sell1-sigma256", 4097), ("vi4-256", 129),
               ("diag-7-254", 4097), ("diag-32-254", 129), ("boundary-fuse1", 4097)]
SMOOTHERS = {"jacobi": {}, "l1jacobi": {"smoother": "l1jacobi"}, "cheb1": {"smoother": "chebyshev", "cheb_degree": 1},
             "cheb2": {"smoother": "chebyshev", "cheb_degree": 2}}


@need_ld
@pytest.mark.gpu
@pytest.mark.parametrize("smoother", sorted(SMOOTHERS))
@pytest.mark.parametrize("name,n", SMOOTH_GRID, ids=[f"{c}-n{n}" for c, n in SMOOTH_GRID])
def test_smoother_rows(name, n, smoother, monkeypatch):
    """One sweep x+ of pamg_smooth, every row within its bound (w, dinv, c1, c2 are the fp64 numbers the library computes).
    Jacobi / l1-Jacobi, x+ = x + w (b - s): |x+^ - x+| <= gamma_{k+3} (|x| + |w| (|b| + S)), S = sum_j |a_ij x_j| (the sum, b - s,
    w * (.), x + (.): k + 3 roundings, fewer when contracted).
    Chebyshev step 1 (c1 multiplies a zero): d = c2 (dinv (b - s)), x+ = x + d: |d^ - d| <= gamma_{k+3} |c2 dinv| (|b| + S) =: Ed,
    |x+^ - x+| <= gamma_{k+4} (|x| + |c2 dinv| (|b| + S)) =: Ex.
    Chebyshev degree 2, step 2 from the computed x1^, d1^: d2 = c1 d1 + c2 dinv (b - A x1), x2 = x1 + d2.  The rounding of step 2
    itself is within gamma_{k+5} (|x1^| + |c1 d1^| + |c2 dinv| (|b| + sum_j |a_ij x1^_j|)); the error of step 1 is carried through
    as Ex_i + |c1| Ed_i + |c2 dinv_i| sum_j |a_ij| Ex_j, with |x1^| <= |x1| + Ex and |d1^| <= |d1| + Ed."""
    s = case(name, n)
    oopts = SMOOTHERS[smoother]
    gh = s["h"]["global"]
    h = hierarchy(gh["levels"][0]["A"], gh["levels"][0]["P"], gh["levels"][0]["owner"], gh["levels"][1]["owner"], s["nparts"], oopts)
    c = device_context(s, monkeypatch, oopts, h)
    lev0 = h["levels"][0]
    A = gh["levels"][0]["A"]
    b, x0 = det_vector(n, 21), det_vector(n, 22)
    c.pcg(own_parts(lev0, b), maxiter=1)
    fam, names = launch_families(c)
    mode = "cheb" if smoother.startswith("cheb") else "jacobi+dot"             # the last post-smoothing sweep carries r . z
    assert fam.get(("A0", mode)) == s["want"][("A0", "resid")], (fam, names)
    got = gather(lev0, c.smooth(0, 1, own_parts(lev0, b), own_parts(lev0, x0)), n)
    diag, diag_l1 = np.zeros(n), np.zeros(n)
    for p, d in enumerate(lev0["parts"]):
        diag[d["own_to_global"]], diag_l1[d["own_to_global"]] = c.diag(0, p)
    bl, xl = b.astype(LD), x0.astype(LD)
    s0, S0, k = ext_rows([(A, x0)], n)
    rows = np.arange(n)
    what = f"{name} n={n} {smoother}"
    if mode != "cheb":
        w = (1.0 / diag_l1 if smoother == "l1jacobi" else (2.0 / 3.0) / diag).astype(LD)
        ref = xl + w * (bl - s0)
        assert_bounded(what, rows, got, ref, gamma2(k + 3) * (np.abs(xl) + np.abs(w) * (np.abs(bl) + S0)))
        return
    rho = h["rho_dinv_a"][0]                                  # engine.cu enqueue_smooth, in the library's fp64 operations
    lmax, lmin = 1.0 * rho, (1.0 / 30.0) * rho
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    sigma = theta / delta
    dinv = (1.0 / diag).astype(LD)
    cw = LD(1.0 / theta) * dinv
    d1 = cw * (bl - s0)
    x1 = xl + d1
    Ed = gamma2(k + 3) * np.abs(cw) * (np.abs(bl) + S0)
    Ex = gamma2(k + 4) * (np.abs(xl) + np.abs(cw) * (np.abs(bl) + S0))
    if smoother == "cheb1":
        assert_bounded(what, rows, got, x1, Ex)
        return
    rho_k = 1.0 / sigma
    rho_n = 1.0 / (2.0 * sigma - rho_k)
    c1, c2 = LD(rho_n * rho_k), LD(2.0 * rho_n / delta)
    s1, _, _ = ext_rows([(A, x1)], n)
    x1_abs = np.abs(x1) + Ex
    _, S1, _ = ext_rows([(A, x1_abs)], n)                     # sum_j |a_ij| |x1^_j|
    _, AEx, _ = ext_rows([(A, Ex)], n)
    d2 = c1 * d1 + c2 * dinv * (bl - s1)
    ref = x1 + d2
    local = gamma2(k + 5) * (x1_abs + abs(c1) * (np.abs(d1) + Ed) + np.abs(c2 * dinv) * (np.abs(bl) + S1))
    carried = Ex + abs(c1) * Ed + np.abs(c2 * dinv) * AEx
    assert_bounded(what, rows, got, ref, local + carried)


# ---- GPU: launches that stride over the slices more than once -----------------------------------------------------------------
@functools.lru_cache(maxsize=1)
def _large(n):
    A = stencil(n, [-(n // 2), -1024, -1, 0, 1, 1024, n // 2], 254)
    owner = np.zeros(n, np.int32)
    P, cown = prolongator(A, owner, 1000)
    return hierarchy(A, P, owner, cown, 1)


@need_ld
@pytest.mark.gpu
@pytest.mark.timeout(900, method="thread")
@pytest.mark.parametrize("fmt", ["sell-vi", "sell-diag"])
def test_multi_pass_launches(fmt):
    """The bounded launches (one resident wave, mean row length <= 12) stride over the slices: the look-ahead of the 128-row
    value-indexed kernel and the implied-column kernel's loop.  A wave holds at most min(RED_GRID, 8 CTAs/SM) CTAs of 256 threads
    (2048 threads per SM), 8 warps per CTA, one 128-row slice per warp and pass: twice that many slices plus a partial one make
    every warp take at least two passes."""
    import torch
    pr = torch.cuda.get_device_properties(0)
    ctas = min(RED_GRID, pr.max_threads_per_multi_processor // 256 * pr.multi_processor_count)
    n = 2 * ctas * 8 * SLICE_ROWS + 77
    assert -(-n // SLICE_ROWS) > 2 * ctas * 8
    h = _large(n)
    opts = dict(spmv_format=L.FORMAT_SELL, sell_sigma=1) if fmt == "sell-vi" else dict(spmv_format=L.FORMAT_SELL_DIAG)
    c = product_context_from_oracle(h, None, **opts)
    c.device_init()
    lev0 = h["levels"][0]
    b = det_vector(n, 5)
    check_cg_step(f"{fmt} n={n} CG", c, h, b, precond=False)
    fam, names = launch_families(c)
    assert fam[("A0", "mul+dot")] == fmt, names
    assert vi_bits_ok(fmt, c.stats().value_indexed[0])
    for seed, xv in ((1, det_vector(n, 11)), (2, 1.0 + 2.0 ** -30 * det_vector(n, 12))):
        check_op(f"{fmt} x{seed} A x", h, "A", xv, c.spmv(0, [xv]), fmt)
        bv = h["global"]["levels"][0]["A"] @ xv
        r, bc = c.residual_restrict(0, [bv], [xv])
        check_op(f"{fmt} x{seed} b - A x", h, "A", xv, r, fmt, "resid", bv)
    c.close()
