"""GPU tests of the compact 5-plane PNP Jacobian (planes L, M, (c+,phi), (c-,phi), D; pnp_block<5>()) and of every
solver kernel that reads it, against references that do not share the device's code:

  * entries: the compact Jacobian of a user matrix (pnp_tune "matrix_compact" = 1) exported and compared with the CPU
    oracle's exact derivative, plus the structure the layout implies (unit Dirichlet rows, exact zeros, bit-identical
    planes shared with the 7-plane layout);
  * SpMV: pnp_spmv with 5 planes, plain-load and streaming kernels, against an exact-sum product of the exported matrix;
  * Jacobi: the stored reciprocal of the rounded diagonal, bit for bit;
  * one smoother step (damped point-block Jacobi, Chebyshev) of the multigrid against a numpy restatement with a
    propagated rounding bound, with 5 and with 7 planes;
  * whole multigrid cycles, compact against 7 planes, over a pairwise cover of the multigrid options;
  * the Newton / linear-problem work space (no knob): its SpMV byte counters show 5 planes (7 where the layout does not
    apply), and the step solves the oracle's system row by row;
  * refusals: FD assembly, SSOR, ILU0, the Gauss-Seidel smoother and CSR import refuse a compact matrix.

Rounding notation: u = 2^-53, gamma(n) = n u / (1 - n u), the bound of n roundings in a sum or dot product.
"""
import itertools
import math

import numpy as np
import pytest
import scipy.sparse as sp

import util
from oracle import binding as ora
from test_gpu_compact_jacobian import mixed_cfg
from test_gpu_parity import TOL_EXACT, rel_err

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
TMA_TR, TMA_CAP = 128, 960  # rows per tile and staged slots per tile of the streaming SpMV (pnp_spmv_tma.cuh)
DEFAULT_TUNE = dict(matrix_compact=0, jac_compact=1, tma_min_rows=-1, tma_lpr=2, tma_stages=2)


def gamma(n):
    n = np.asarray(n, dtype=np.float64)
    return n * U / (1.0 - n * U)


def _capi():
    from dune_pnp_b200 import capi
    return capi


@pytest.fixture
def knobs():
    capi = _capi()

    def set_(**kw):
        for k, v in kw.items():
            capi.tune(k, v)
    yield set_
    for k, v in DEFAULT_TUNE.items():
        capi.tune(k, v)


def fan_mesh(n=1001):
    """A disc of n triangles around one hub vertex (one_wall.cfg's surfaces 1 and 0 on the two halves of the rim): the
    hub's star row has n + 1 slots, so the streaming SpMV's first tile is over-full (plain-load fallback)."""
    t = 2.0 * np.pi * np.arange(n) / n
    x = np.concatenate([[5.0], 5.0 + 3.0 * np.cos(t)])
    y = np.concatenate([[5.0], 5.0 + 3.0 * np.sin(t)])
    rim = 1 + np.arange(n)
    nxt = 1 + (np.arange(n) + 1) % n
    tri = np.stack([np.zeros(n, dtype=np.int32), rim, nxt], axis=1).astype(np.int32)
    return dict(x=x, y=y, tri=tri, ba=rim.astype(np.int32), bb=nxt.astype(np.int32),
                bphys=(np.arange(n) < n // 2).astype(np.int32))


def make_ctx(name, levels=0, renumber=True, cfg=None, oracle=True):
    capi = _capi()
    a = fan_mesh() if name == "fan" else util.load_mesh_arrays(name)
    cfg = cfg or util.cfg_path("one_wall" if name == "fan" else name)
    c = capi.Context(0)
    c.mesh_set(**a)
    c.params_read(cfg)
    if levels:
        c.mesh_refine(levels)
    c.mesh_finalize(renumber)
    if not oracle:
        return c, None, None
    return c, ora.Mesh.from_arrays(**a).refine(levels), ora.Params.read(cfg)


# ---- states (reference numbering, fields concatenated: phi, c+, c-) ----
def smooth_state(x, y):
    sx, sy = np.ptp(x), np.ptp(y)
    return np.concatenate([5.0 * np.sin(2.0 * x / sx) * np.cos(y / sy), 0.06 * (1.0 + 0.3 * np.cos(3.0 * y / sy)),
                           0.06 * (1.0 - 0.2 * np.sin(2.0 * x / sx + y / sy))])


def newton_state(x, y):
    """phi in +-30 and concentrations in [0, 2): large drift D and phi/c couplings, as in an early Newton iterate."""
    rng = np.random.RandomState(1)
    n = len(x)
    return np.concatenate([rng.uniform(-30, 30, n), rng.uniform(0, 2, n), rng.uniform(0, 2, n)])


def zero_c_state(x, y):
    """the smooth state with both concentrations exactly 0 on the left half of the mesh (the drift D vanishes there)"""
    u = smooth_state(x, y).reshape(3, -1).copy()
    u[1:, x < np.median(x)] = 0.0
    return u.ravel()


STATES = {"smooth": smooth_state, "newton": newton_state, "zero_c": zero_c_state}


def assembled(c, h, u, compact, knobs):
    """a user matrix of the PNP operator (5 planes where the knob gives them, else 7) assembled at u, exact derivative"""
    capi = _capi()
    knobs(matrix_compact=1 if compact else 0)
    A = c.matrix(h)
    c.jacobian(h, c.vec(3, u), A, capi.JAC_ANALYTIC, 0.0)
    return A


def export(c, h, A):
    rp, col = c.pattern(h, 3)
    return rp, col, c.matrix_values(h, A, len(col))


def entry_fields(rp, col, nv):
    row = np.repeat(np.arange(len(rp) - 1, dtype=np.int64), np.diff(rp))
    return row, (row // nv).astype(np.int8), (col // nv).astype(np.int8)


def diag_blocks(rp, col, val, nv):
    """the 3x3 diagonal block of every vertex (reference numbering) from an exported PNP matrix"""
    row, ki, kj = entry_fields(rp, col, nv)
    same = (row % nv) == (col % nv)
    B = np.zeros((nv, 3, 3))
    B[row[same] % nv, ki[same], kj[same]] = val[same]
    return B


# ---------------------------------------------------------------------------------------------------------------------
# 1. entries
ENTRY_CASES = ([(n, 0, s) for n in util.MESHES for s in STATES] + [(n, 2, s) for n in ("pore_small", "one_wall") for s in STATES]
               + [("pore", 4, "newton")])


@pytest.mark.parametrize("name,levels,state", ENTRY_CASES)
def test_compact_entries_match_the_oracle(name, levels, state, knobs):
    """Compact export against the oracle's exact derivative within TOL_EXACT of the per-entry scale, and the structure the
    layout implies.  pore at level 4 (780 k vertices) runs the Newton-like state only, for the staging tiles of the
    assembly kernel at size.  The compact and 7-plane diagonal blocks group the element contributions differently
    ((L - D) summed once against L and D summed apart), so they agree to 8 ulp of the sum of the absolute element
    contributions of L and D -- the oracle's per-entry scales of (phi,phi), (c+,c+) and (c-,c-) -- not bit for bit."""
    capi = _capi()
    c, m, p = make_ctx(name, levels)
    nv = m.nv
    u = STATES[state](m.x, m.y)
    h = c.operator(capi.OP_PNP, 0)
    rp, col, val_o, ab = ora.jacobian(m, p, ora.OP_PNP, u, mode=1, want_abs=True)
    v5 = export(c, h, assembled(c, h, u, True, knobs))[2]
    v7 = export(c, h, assembled(c, h, u, False, knobs))[2]
    assert rel_err(v5, val_o, ab) <= TOL_EXACT
    del val_o
    row, ki, kj = entry_fields(rp, col, nv)
    d = ora.dirichlet(m, p, 3)
    assert np.array_equal(d[:nv], d[nv:2 * nv]) and np.array_equal(d[:nv], d[2 * nv:])  # the layout's precondition
    dr = d[row]
    assert np.array_equal(v5[dr], (col[dr] == row[dr]).astype(np.float64))  # unit Dirichlet rows
    assert not np.any(v5[d[col] & (col != row)])                               # zero Dirichlet columns
    cross = ((ki == 1) & (kj == 2)) | ((ki == 2) & (kj == 1))
    assert cross.any() and np.all(v5[cross] == 0.0)
    for a, b in ((0, 0), (0, 1), (1, 0), (2, 0)):
        s = (ki == a) & (kj == b)
        assert np.array_equal(v5[s], v7[s]), (a, b)
    key = (row % nv) * nv + col % nv
    blk = {(a, b): (ki == a) & (kj == b) for a, b in ((0, 0), (0, 1), (0, 2), (1, 1), (2, 2))}
    assert np.array_equal(key[blk[0, 1]], key[blk[0, 2]]) and np.array_equal(v5[blk[0, 2]], -v5[blk[0, 1]])
    assert np.array_equal(key[blk[0, 0]], key[blk[1, 1]]) and np.array_equal(key[blk[0, 0]], key[blk[2, 2]])
    scale = ab[blk[0, 0]] + ab[blk[1, 1]] + ab[blk[2, 2]]
    for s in (blk[1, 1], blk[2, 2]):
        assert np.all(np.abs(v5[s] - v7[s]) <= 8 * np.spacing(scale))


# ---------------------------------------------------------------------------------------------------------------------
# 2. SpMV
SPMV_MESHES = [("one_wall", 0), ("sphere", 0), ("pore_without_dna", 0), ("pore_small", 2), ("fan", 0)]
SPMV_SETTINGS = [(-1, 2, 2)] + [(1, lpr, st) for lpr in (1, 2) for st in (2, 3)]  # (tma_min_rows, tma_lpr, tma_stages)


def star_row_lengths(g, renumber):
    """slots of every star row in the kernels' row order: the diagonal and one per neighbour; with the locality
    renumbering rows are ordered by the first triangle corner that touches them (pnp_setup.cu, star_build)"""
    tri = g["tri"].astype(np.int64)
    nv = len(g["x"])
    e = np.sort(np.concatenate([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]]), axis=1)
    deg = np.bincount(np.unique(e, axis=0).ravel(), minlength=nv)
    order = np.arange(nv)
    if renumber:
        first = np.full(nv, np.iinfo(np.int64).max)
        np.minimum.at(first, tri.ravel(), np.arange(tri.size))
        order = np.argsort(first, kind="stable")
    return 1 + deg[order]


def two_prod(a, b):
    """a*b = p + e exactly (Veltkamp / Dekker)"""
    p = a * b
    f = 134217729.0
    ah = a * f; ah = ah - (ah - a); al = a - ah
    bh = b * f; bh = bh - (bh - b); bl = b - bh
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


@pytest.mark.parametrize("renumber", [True, False])
def test_compact_spmv_within_the_exact_sum_bound(renumber, knobs):
    """y = A x of a compact matrix against the correctly rounded exact sum of the exported row (math.fsum of exact
    products): |y - y_ref| <= gamma(n) sum|a_ij x_j| + u |y_ref| per row, n = the row's terms.  Plain-load kernel and
    streaming kernel (tma_min_rows = 1) with 1 and 2 lanes per row and 2 and 3 stages.  The cases must contain a mesh
    with fewer than 128 vertices, one with a partial last tile, odd nslots (the plane-parity offset of the bulk copies),
    an over-full tile and rows of more than 8 slots; these are computed from the star of each mesh built here."""
    capi = _capi()
    shapes = set()
    for name, levels in SPMV_MESHES:
        c, _, _ = make_ctx(name, levels, renumber, oracle=False)
        g = c.mesh_get()
        sz = c.mesh_sizes()
        nv, ns = sz["nv"], sz["nslots"]
        L = star_row_lengths(g, renumber)
        assert L.sum() == ns
        tiles = np.add.reduceat(L, np.arange(0, nv, TMA_TR))
        shapes |= {s for s, on in (("nv<128", nv < TMA_TR), ("partial tile", nv % TMA_TR != 0), ("odd nslots", ns % 2 == 1),
                                   ("over-full tile", tiles.max() > TMA_CAP), ("rows>8", L.max() > 8)) if on}
        h = c.operator(capi.OP_PNP, 0)
        A = assembled(c, h, newton_state(g["x"], g["y"]), True, knobs)
        rp, col, val = export(c, h, A)
        x = np.random.RandomState(11).uniform(-1, 1, 3 * nv)
        p, e = two_prod(val, x[col])
        y_ref = np.array([math.fsum(np.concatenate([p[a:b], e[a:b]])) for a, b in zip(rp[:-1], rp[1:])])
        S = np.add.reduceat(np.abs(p), rp[:-1])
        bound = gamma(np.diff(rp)) * S + U * np.abs(y_ref)
        vx, vy = c.vec(3, x), c.vec(3)
        for min_rows, lpr, stages in SPMV_SETTINGS:
            knobs(tma_min_rows=min_rows, tma_lpr=lpr, tma_stages=stages)
            c.vec_set(vy, np.nan)
            c.spmv(A, vx, vy)
            y = c.download(vy, 3)
            assert np.all(np.abs(y - y_ref) <= bound), (name, min_rows, lpr, stages, np.max(np.abs(y - y_ref) - bound))
    assert shapes == {"nv<128", "partial tile", "odd nslots", "over-full tile", "rows>8"}, shapes


# ---------------------------------------------------------------------------------------------------------------------
# 3. Jacobi
@pytest.mark.parametrize("name,levels", [(n, 0) for n in util.MESHES] + [("pore_small", 2)])
def test_compact_jacobi_is_the_reciprocal_of_the_exported_diagonal(name, levels, knobs):
    """PREC_JACOBI stores 1/(L -+ D) of the same rounded L -+ D the export shows and multiplies: bit for bit."""
    capi = _capi()
    c, _, _ = make_ctx(name, levels, oracle=False)
    g = c.mesh_get()
    nv = len(g["x"])
    h = c.operator(capi.OP_PNP, 0)
    A = assembled(c, h, newton_state(g["x"], g["y"]), True, knobs)
    rp, col, val = export(c, h, A)
    row = np.repeat(np.arange(3 * nv), np.diff(rp))
    on = col == row
    diag = np.full(3 * nv, np.nan)
    diag[row[on]] = val[on]
    dvec = np.random.RandomState(5).uniform(-1, 1, 3 * nv)
    vd, vv = c.vec(3, dvec), c.vec(3)
    c.precond_apply(c.solver(capi.SOLVER_BCGS, capi.PREC_JACOBI), A, vd, vv)
    assert np.array_equal(c.download(vv, 3), (1.0 / diag) * dvec)


# ---------------------------------------------------------------------------------------------------------------------
# 4. one smoother step
def block_inverse(B):
    """k_dinv / block_inverse_row restated: cofactor inverse of [a b c; d e 0; f 0 g], scalar diagonal where
    |det| <= 1e-12 scale.  Returns the inverse, a bound of its rounding (8 u (1 + scale/|det|) times the absolute
    cofactors over |det|: det and the cofactors are sums of three and two products), the fallback vertices and
    |det| / scale."""
    a, b, c_, d, e, f, g = (B[:, 0, 0], B[:, 0, 1], B[:, 0, 2], B[:, 1, 0], B[:, 1, 1], B[:, 2, 0], B[:, 2, 2])
    det = a * e * g - b * d * g - c_ * e * f
    scale = np.abs(a * e * g) + np.abs(b * d * g) + np.abs(c_ * e * f)
    ok = (np.abs(det) > 1e-12 * scale) & (scale > 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        idet = 1.0 / det
        cof = np.stack([e * g, -b * g, -c_ * e, -d * g, a * g - c_ * f, c_ * d, -e * f, b * f, a * e - b * d], axis=1)
        cabs = np.stack([np.abs(e * g), np.abs(b * g), np.abs(c_ * e), np.abs(d * g), np.abs(a * g) + np.abs(c_ * f),
                         np.abs(c_ * d), np.abs(e * f), np.abs(b * f), np.abs(a * e) + np.abs(b * d)], axis=1)
        Dinv = (cof * idet[:, None]).reshape(-1, 3, 3)
        E = (8 * U * (1.0 + scale / np.abs(det))[:, None] * cabs / np.abs(det)[:, None]).reshape(-1, 3, 3)
        ratio = np.where(scale > 0, np.abs(det) / scale, 1.0)
    for k, dd in enumerate((a, e, g)):  # fallback: the scalar diagonal
        inv = np.where(dd != 0.0, 1.0 / np.where(dd != 0.0, dd, 1.0), 0.0)
        Dinv[~ok, k, :] = 0.0; E[~ok, k, :] = 0.0
        Dinv[~ok, k, k] = inv[~ok]; E[~ok, k, k] = U * np.abs(inv[~ok])
    return Dinv, E, ~ok, ratio


def bapply(M, r):
    """z[k*nv + v] = sum_j M[v, k, j] r[j*nv + v]"""
    return np.einsum("vkj,jv->kv", M, r.reshape(3, -1)).ravel()


def smoother_reference(A, Dinv, E, b, nu, smoother, lmax=None, omega=0.7, ratio=8.0):
    """nu steps of the multigrid smoother from x = 0 (pnp_amg.cu, smooth()) and a bound of the rounding of any float64
    evaluation of the same recurrence (device or this one): r = b - A x within gamma(n + 1)(|b| + |A||x|); z = M^-1 r
    within E|r| + |M^-1| dr + gamma(4)|M^-1||r| (three-term dot and the damping product); each update one or two
    additions."""
    Aabs = abs(A)
    nrow = np.diff(A.indptr).max()
    Dabs = np.abs(Dinv) + E
    gr, g4 = gamma(nrow + 1), gamma(4)

    def z_err(rabs, dr):
        return bapply(E, rabs) + bapply(Dabs, dr) + g4 * bapply(Dabs, rabs)
    if smoother == 0:
        x = omega * bapply(Dinv, b)
        dx = omega * z_err(np.abs(b), 0.0 * b)
        for _ in range(1, nu):
            rabs = np.abs(b) + Aabs @ np.abs(x)
            z = bapply(Dinv, b - A @ x)
            dz = z_err(rabs, gr * rabs + Aabs @ dx)
            dx = dx + omega * dz + 2 * U * (np.abs(x) + omega * np.abs(z))
            x = x + omega * z
        return x, dx
    lmx, lmn = 1.1 * lmax, lmax / ratio
    theta, delta = 0.5 * (lmx + lmn), 0.5 * (lmx - lmn)
    sigma = theta / delta
    rho = 1.0 / sigma
    x = (1.0 / theta) * bapply(Dinv, b)
    dx = (1.0 / theta) * z_err(np.abs(b), 0.0 * b)
    dvec, dd = x.copy(), dx.copy()
    for _ in range(1, nu):
        rho_new = 1.0 / (2.0 * sigma - rho)
        c2, c1 = 2.0 * rho_new / delta, rho_new * rho
        rabs = np.abs(b) + Aabs @ np.abs(x)
        z = bapply(Dinv, b - A @ x)
        dz = z_err(rabs, gr * rabs + Aabs @ dx)
        dvec_new = c1 * dvec + c2 * z
        dd = c1 * dd + c2 * dz + 3 * U * (c1 * np.abs(dvec) + c2 * np.abs(z))
        dx = dx + dd + U * (np.abs(x) + np.abs(dvec_new))
        x, dvec = x + dvec_new, dvec_new
        rho = rho_new
    return x, dx


@pytest.mark.parametrize("planes", [5, 7])
@pytest.mark.parametrize("min_rows", [1, -1])
@pytest.mark.parametrize("smoother", [0, 1])
def test_one_smoother_step_matches_numpy(smoother, min_rows, planes, knobs):
    """precond_apply(PREC_AMG) with nu pre-smoothing steps, no post-smoothing, amg_alpha = 0 (no coarse correction on the
    algebraic levels of this unrefined mesh) and no dense coarse solve is nu smoother steps on the fine level.  Damped
    point-block Jacobi (tma_min_rows = 1: the streaming kernel inverts each diagonal block itself; default: the plain
    kernel reads the stored k_dinv inverse) and Chebyshev (always the plain kernel) against the numpy recurrence within
    twice the rounding bound of smoother_reference.  Chebyshev's Gershgorin bound is recomputed here; the device's sum
    differs by its rounding, gamma(n) relative, and the recurrence's spread over lmax (1 +- 2 gamma(n)) is added.
    The Newton-like state has diagonal blocks with |det| / scale below 1e-3, so a looser singularity threshold changes
    the result; no block of a legitimate state comes near 1e-12 (fine-level Dirichlet blocks are identities), so no
    vertex takes the scalar fallback, which the reference reports."""
    capi = _capi()
    c, _, _ = make_ctx("pore_without_dna", 0, oracle=False)
    g = c.mesh_get()
    nv = len(g["x"])
    h = c.operator(capi.OP_PNP, 0)
    A = assembled(c, h, newton_state(g["x"], g["y"]), planes == 5, knobs)
    rp, col, val = export(c, h, A)
    As = sp.csr_matrix((val, col, rp), shape=(3 * nv, 3 * nv))
    Dinv, E, fallback, ratio = block_inverse(diag_blocks(rp, col, val, nv))
    assert not fallback.any() and (ratio < 1e-3).any()
    lmax = None
    if smoother == 1:
        rows = np.add.reduceat(np.abs(val), rp[:-1])
        lmax = np.max(rows / np.abs(As.diagonal()))
        spread_l = 2 * gamma(np.diff(rp).max())
    knobs(tma_min_rows=min_rows)
    b = np.random.RandomState(9).uniform(-1, 1, 3 * nv)
    vb, vy = c.vec(3, b), c.vec(3)
    for nu in (1, 2, 3):
        s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 1, 1)
        for k, v in (("amg_smoother", smoother), ("amg_pre_steps", nu), ("amg_post_steps", 0), ("amg_alpha", 0.0),
                     ("amg_dense_max", 0), ("amg_geometric", 0), ("amg_coarse_sweeps", 0)):
            c.solver_set_option(s, k, v)
        c.precond_apply(s, A, vb, vy)
        y = c.download(vy, 3)
        x, dx = smoother_reference(As, Dinv, E, b, nu, smoother, lmax)
        tol = 2 * dx
        if smoother == 1:
            for lm in (lmax * (1 - spread_l), lmax * (1 + spread_l)):
                tol = tol + np.abs(smoother_reference(As, Dinv, E, b, nu, smoother, lm)[0] - x)
        assert np.all(np.abs(y - x) <= tol), (nu, np.max(np.abs(y - x) - tol))


# ---------------------------------------------------------------------------------------------------------------------
# 5. whole cycles, compact against 7
CYCLE_FACTORS = {"amg_geometric": (0, 1), "amg_rediscretise": (0, 1), "amg_smoother": (0, 1), "amg_gamma": (1, 2),
                 "amg_dense_max": (0, 4096), "tma_min_rows": (-1, 1)}
# Six runs cover every pair of levels of every two factors: the factors' columns are six distinct 6-bit words of weight 3
# with a 0 first bit; any two such words show 00 (first bit), 11 (two 3-subsets of 5 positions meet), 10 and 01.
_WORDS = [w for w in itertools.combinations(range(1, 6), 3)][: len(CYCLE_FACTORS)]
CYCLE_RUNS = [{k: CYCLE_FACTORS[k][int(r in w)] for k, w in zip(CYCLE_FACTORS, _WORDS)} for r in range(6)]
assert all({(run[a], run[b]) for run in CYCLE_RUNS} == set(itertools.product(CYCLE_FACTORS[a], CYCLE_FACTORS[b]))
           for a, b in itertools.combinations(CYCLE_FACTORS, 2))


@pytest.mark.parametrize("name,opts", list(zip(util.MESHES, CYCLE_RUNS)))
def test_multigrid_cycle_compact_equals_seven_planes(name, opts, knobs):
    """One default V(2,2) application (gamma 2: W) on each mesh refined twice, compact against 7 planes assembled at the same
    smooth state, relative difference <= 1e-11.  The six meshes carry a pairwise cover of geometric / pure aggregation
    (k_galerkin with its Dirichlet zeroing), Galerkin / re-discretised geometric levels, Jacobi / Chebyshev smoother
    (k_gershgorin), V / W cycle, no dense / dense coarsest level (k_dense_fill) and the streaming SpMV on every level /
    the default threshold (CYCLE_RUNS)."""
    capi = _capi()
    c, _, _ = make_ctx(name, 2, oracle=False)
    g = c.mesh_get()
    nv = len(g["x"])
    u = smooth_state(g["x"], g["y"])
    knobs(tma_min_rows=opts["tma_min_rows"])
    h = c.operator(capi.OP_PNP, 0)
    dvec = np.random.RandomState(13).uniform(-1, 1, 3 * nv)
    vd = c.vec(3, dvec)
    y = {}
    for planes in (5, 7):
        A = assembled(c, h, u, planes == 5, knobs)  # right before its application: re-discretisation keys on it
        s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 1, 2)
        for k, v in opts.items():
            if k != "tma_min_rows":
                c.solver_set_option(s, k, v)
        vy = c.vec(3)
        c.precond_apply(s, A, vd, vy)
        y[planes] = c.download(vy, 3)
    assert np.all(np.isfinite(y[7])) and np.linalg.norm(y[7]) > 0
    assert np.linalg.norm(y[5] - y[7]) <= 1e-11 * np.linalg.norm(y[7])


# ---------------------------------------------------------------------------------------------------------------------
# 6. the work space
def slp_spmv_bytes(c, h, u0, prec, jac_compact, knobs):
    """fine-level SpMV bytes and launches of two BiCGSTAB iterations of the linear-problem step"""
    capi = _capi()
    knobs(jac_compact=jac_compact)
    c.profile_spmv(True)
    c.profile_bytes(reset=True)
    c.slp(h, c.vec(3, u0), c.solver(capi.SOLVER_BCGS, prec, 2, 1), 1e-30, jac_mode=capi.JAC_ANALYTIC, eps=0.0)
    launches = sum(c.profile_spmv_get()[0])
    c.profile_spmv(False)
    return c.profile_bytes(reset=True)["spmv_fine"], launches


WS_CASES = [(n, "amg") for n in util.MESHES] + [(n, p) for n in ("one_wall", "sphere", "cylinder") for p in ("jacobi", "none")]


@pytest.mark.parametrize("name,prec", WS_CASES)
def test_workspace_reads_five_planes_and_solves_the_oracle_system(name, prec, knobs):
    """The Newton / linear-problem work space with no knob set (multigrid: meshes refined once; Jacobi and no
    preconditioner: the three smallest meshes unrefined).  Bytes: the same two iterations with jac_compact 1 and 0
    launch the same fine-level SpMVs, and the compact run reads 16 B (two planes) less per slot and launch.
    Solve: the step z of slp at reduction 1e-13 satisfies the ORACLE's system row by row,
    |A_o z - r_o| <= 10 red |r_o|_2 (BiCGSTAB stops on a recursively updated residual that drifts from the true one)
    + TOL_EXACT ab_A |z| + 1e-12 ab_r (the device's exact-derivative entries and residual against the oracle's, per-entry
    scales) + gamma(n + 1)(|A_o||z| + |r_o|) (this product).  A wrong work-space entry leaves (A_o - A) z in its row."""
    capi = _capi()
    prec_id = {"amg": capi.PREC_AMG, "jacobi": capi.PREC_JACOBI, "none": capi.PREC_NONE}[prec]
    c, m, p = make_ctx(name, 1 if prec == "amg" else 0)
    u0 = smooth_state(m.x, m.y)
    h = c.operator(capi.OP_PNP, 0)
    ns = c.mesh_sizes()["nslots"]
    b5, l5 = slp_spmv_bytes(c, h, u0, prec_id, 1, knobs)
    b7, l7 = slp_spmv_bytes(c, h, u0, prec_id, 0, knobs)
    assert l5 == l7 and l5 > 0 and b7 - b5 == 16.0 * ns * l5, (b5, b7, l5, l7)
    knobs(jac_compact=1)
    red = 1e-13
    vu = c.vec(3, u0)
    res = c.slp(h, vu, c.solver(capi.SOLVER_BCGS, prec_id, 20000, 1), red, jac_mode=capi.JAC_ANALYTIC, eps=0.0)
    assert res.converged
    z = u0 - c.download(vu, 3)
    rp, col, val_o, ab = ora.jacobian(m, p, ora.OP_PNP, u0, mode=1, want_abs=True)
    r_o, abr = ora.residual(m, p, ora.OP_PNP, u0, want_abs=True)
    N = 3 * m.nv
    Ao, Ab = sp.csr_matrix((val_o, col, rp), shape=(N, N)), sp.csr_matrix((ab, col, rp), shape=(N, N))
    lhs = np.abs(Ao @ z - r_o)
    bound = (10 * red * np.linalg.norm(r_o) + TOL_EXACT * (Ab @ np.abs(z)) + 1e-12 * abr
             + gamma(np.diff(rp) + 1) * (abs(Ao) @ np.abs(z) + np.abs(r_o)))
    assert np.linalg.norm(z) > 0 and np.all(lhs <= bound), np.max(lhs - bound)


def test_workspace_keeps_seven_planes_where_the_layout_does_not_apply(knobs, tmp_path):
    """a surface with a Dirichlet potential and Neumann concentrations: the work space reads the same bytes either way"""
    capi = _capi()
    c, m, _ = make_ctx("pore", 1, cfg=mixed_cfg(tmp_path))
    u0 = smooth_state(m.x, m.y)
    h = c.operator(capi.OP_PNP, 0)
    b_on, l_on = slp_spmv_bytes(c, h, u0, capi.PREC_AMG, 1, knobs)
    b_off, l_off = slp_spmv_bytes(c, h, u0, capi.PREC_AMG, 0, knobs)
    assert l_on == l_off > 0 and b_on == b_off


# ---------------------------------------------------------------------------------------------------------------------
# 7. refusals
def test_compact_user_matrix_refusals(knobs, tmp_path):
    capi = _capi()
    c, m, _ = make_ctx("pore_small", 1, oracle=True)
    u = newton_state(m.x, m.y)
    h = c.operator(capi.OP_PNP, 0)
    A = assembled(c, h, u, True, knobs)
    rp, col, before = export(c, h, A)

    def refused(fn, msg):
        with pytest.raises(capi.PnpError) as e:
            fn()
        assert e.value.status == 8 and msg in str(e.value), str(e.value)
    refused(lambda: c.jacobian(h, c.vec(3, u), A, capi.JAC_FD_FAITHFUL, 1e-11), "matrix layout does not fit")
    vd, vv = c.vec(3, u), c.vec(3)
    for prec, opts, msg in ((capi.PREC_SSOR, {}, "SSOR sweeps 7-plane PNP matrices only"),
                            (capi.PREC_ILU0, {}, "ILU0 factors 7-plane PNP matrices only"),
                            (capi.PREC_AMG, {"amg_smoother": 2}, "Gauss-Seidel smoother sweeps 7-plane PNP matrices only")):
        s = c.solver(capi.SOLVER_BCGS, prec)
        for k, v in opts.items():
            c.solver_set_option(s, k, v)
        refused(lambda: c.precond_apply(s, A, vd, vv), msg)
    refused(lambda: c.matrix_set_csr(h, A, rp, col, before), "matrix import writes the 7-plane PNP layout only")
    assert np.array_equal(export(c, h, A)[2], before)
    # where the layout does not apply the knob gives 7 planes: import, FD assembly and export work
    c2, m2, _ = make_ctx("pore_small", 1, cfg=mixed_cfg(tmp_path))
    h2 = c2.operator(capi.OP_PNP, 0)
    u2 = newton_state(m2.x, m2.y)
    A2 = assembled(c2, h2, u2, True, knobs)
    rp2, col2, v_on = export(c2, h2, A2)
    v_off = export(c2, h2, assembled(c2, h2, u2, False, knobs))[2]
    assert np.array_equal(v_on, v_off)
    c2.matrix_set_csr(h2, A2, rp2, col2, v_on)
    c2.jacobian(h2, c2.vec(3, u2), A2, capi.JAC_FD_FAITHFUL, 1e-11)
