"""GPU tests on the hub meshes of util.SHAPES against the CPU oracle: the shapes that reach the kernels' capacity
fallbacks, which the shipped meshes never do (tests/test_host_mesh_shapes.py asserts which shape reaches which):

  * k_jacobian's direct-write path (128-row chunks above JAC_CAP slots) for every exact Jacobian, the compact 5-plane
    export and the multigrid's re-discretised coarse operators;
  * k_jacobian_fdw's per-vertex path (64-row chunks above FDW_CAP slots, rings longer than FDW_KMAX);
  * the streaming SpMV's over-full tiles (above TMA_CAP slots), on a mesh with more tiles than a B200 has SMs;
  * both triangle orientations in one vertex's ring and boundary segments reversed against their element, for the
    element-order reconstruction (FD Jacobian, boundary faces, quadratic and cubic edge dofs).

Tolerances are the shipped meshes' (TOL, TOL_EXACT of test_gpu_parity).  Lines starting with "FIGURE" report the
largest errors observed (pytest -s shows them)."""
import math

import numpy as np
import pytest

import util
from oracle import binding as ora
from test_gpu_compact_layout import DEFAULT_TUNE, U, gamma, two_prod
from test_gpu_p2 import DEG_ORDER
from test_gpu_parity import OPS, TOL, TOL_EXACT, rel_err

pytestmark = pytest.mark.gpu

BASE = [n for n in util.SHAPES if util.SHAPES[n][1] == 0]   # unrefined shapes
ALL = list(util.SHAPES)
TUNE = dict(DEFAULT_TUNE, tma=1, fd_warp=1)


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
    for k, v in TUNE.items():
        capi.tune(k, v)


@pytest.fixture(scope="module")
def cfgs(tmp_path_factory):
    d = tmp_path_factory.mktemp("cfg")
    return {cyl: util.shape_cfg(str(d / ("hub%d.cfg" % cyl)), cyl) for cyl in (0, 1)}


def make_ctx(name, cfg, renumber=True, levels=None, degree=1):
    capi = _capi()
    a, lv = util.shape_arrays(name)
    lv = lv if levels is None else levels
    c = capi.Context(0)
    c.mesh_set(**a)
    c.params_read(cfg)
    if lv:
        c.mesh_refine(lv)
    if degree > 1:
        c.space_set_degree(degree)
    c.mesh_finalize(renumber)
    return c, ora.Mesh.from_arrays(**a).refine(lv), ora.Params.read(cfg)


def _state(m, op, seed):
    """potential and concentrations of an early Newton iterate (concentrations positive)"""
    rng = np.random.RandomState(seed)
    F = ora.nfields(op)
    u = rng.uniform(-1, 1, F * m.nv)
    if op == ora.OP_PNP:
        u[m.nv:] = rng.uniform(0.02, 0.1, 2 * m.nv)
    return u, rng.uniform(0, 1, m.nv), rng.uniform(0, 1, m.nv)


def _operator(c, op, a0, a1, valency=-1.0):
    capi = _capi()
    h = c.operator(op, 0)
    if op == capi.OP_POISSON:
        c.operator_set_coefficient(h, 0, c.vec(1, a0)); c.operator_set_coefficient(h, 1, c.vec(1, a1))
    if op == capi.OP_DIFFUSION:
        c.operator_set_coefficient(h, 0, c.vec(1, a0)); c.operator_set_valency(h, valency)
    return h


def _jacobian(c, m, op, mode, seed=3):
    """device Jacobian values in the oracle's pattern, the oracle's values and per-entry scales"""
    F = ora.nfields(op)
    u, a0, a1 = _state(m, op, seed)
    h = _operator(c, op, a0, a1)
    A = c.matrix(h)
    c.jacobian(h, c.vec(F, u), A, mode, 1e-11 if mode == 0 else 0.0)
    rp, col = c.pattern(h, F)
    return h, A, rp, col, c.matrix_values(h, A, len(col)), (u, a0, a1)


# ---------------------------------------------------------------------------------------------------------------------
# mesh
@pytest.mark.parametrize("name", BASE)
def test_mesh_roundtrip_and_device_refinement(name, cfgs):
    a, _ = util.shape_arrays(name)
    for levels in (0, 1, 2):
        c, m, _ = make_ctx(name, cfgs[1], levels=levels)
        g = c.mesh_get()
        want = a if levels == 0 else dict(x=m.x, y=m.y, tri=m.tri, ba=m.ba, bb=m.bb, bphys=m.bphys)
        for k in want:
            assert np.array_equal(g[k], want[k]), (levels, k)


@pytest.mark.parametrize("renumber", [False, True])
@pytest.mark.parametrize("name", ALL)
def test_pattern_and_constraints_bit_exact(name, renumber, cfgs):
    capi = _capi()
    c, m, p = make_ctx(name, cfgs[1], renumber)
    for F, op, comp0 in ((1, capi.OP_PB, 0), (1, capi.OP_DIFFUSION, 2), (3, capi.OP_PNP, 0)):
        h = c.operator(op, comp0)
        assert np.array_equal(c.constraints(h, F), ora.dirichlet(m, p, F, comp0))
        rp, col = c.pattern(h, F)
        rp_o, col_o = ora.pattern(m, p, F, comp0)
        assert np.array_equal(rp, rp_o) and np.array_equal(col, col_o)


# ---------------------------------------------------------------------------------------------------------------------
# residual and Jacobians
@pytest.mark.parametrize("cylindrical", [0, 1])
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", ALL)
def test_residual_parity(name, op, cylindrical, cfgs):
    """All five operators; alpha_boundary runs on reversed segments and on the open hub fan (non-zero fluxes of all
    three components on surfaces 1 and 3).  Constrained entries are exact zeros."""
    c, m, p = make_ctx(name, cfgs[cylindrical])
    F = ora.nfields(op)
    u, a0, a1 = _state(m, op, 0)
    h = _operator(c, op, a0, a1)
    vr = c.vec(F)
    c.residual(h, c.vec(F, u), vr)
    r = c.download(vr, F)
    r_o, ab = ora.residual(m, p, op, u, a0, a1, valency=-1.0, want_abs=True)
    err = rel_err(r, r_o, ab)
    print("FIGURE residual %s op=%d cyl=%d max_rel=%.3g" % (name, op, cylindrical, err))
    assert err <= TOL
    d = ora.dirichlet(m, p, F, 0)
    assert not r[d].any() and not r_o[d].any()


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", ALL)
def test_fd_jacobian_parity_and_bit_equal_couplings(name, op, cfgs):
    """FD-faithful Jacobian within TOL, and every vertex-coupling (off-diagonal) entry -- a two-term sum of the elements
    on either side of the edge -- bit-equal to the oracle, as the host harness shows for the same functions."""
    c, m, p = make_ctx(name, cfgs[1])
    _, _, rp, col, val, (u, a0, a1) = _jacobian(c, m, op, 0)
    _, _, val_o, ab = ora.jacobian(m, p, op, u, a0, a1, valency=-1.0, mode=0, eps=1e-11, want_abs=True)
    rows = np.repeat(np.arange(len(rp) - 1), np.diff(rp))
    off = (rows % m.nv) != (col % m.nv)
    err, same = rel_err(val, val_o, ab), np.mean(val[off] == val_o[off])
    print("FIGURE fd_jacobian %s op=%d max_rel=%.3g offdiag_bit_equal=%.6f" % (name, op, err, same))
    assert err <= TOL
    assert np.array_equal(val[off], val_o[off]), np.flatnonzero(val[off] != val_o[off])[:10]


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", ALL)
def test_fd_warp_kernel_equals_one_thread_kernel(name, op, cfgs, knobs):
    """fd_warp 1 (warp kernel, per-vertex path for over-full chunks and long rings) against 0 (one thread per vertex,
    staged or direct-write): identical bits."""
    capi = _capi()
    c, m, _ = make_ctx(name, cfgs[1])
    F = ora.nfields(op)
    u, a0, a1 = _state(m, op, 13)
    h = _operator(c, op, a0, a1)
    vu, A = c.vec(F, u), c.matrix(h)
    rp, col = c.pattern(h, F)
    out = {}
    for warp in (1, 0):
        knobs(fd_warp=warp)
        c.jacobian(h, vu, A, capi.JAC_FD_FAITHFUL, 1e-11)
        out[warp] = c.matrix_values(h, A, len(col))
    assert np.array_equal(out[1], out[0])


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", ALL)
def test_exact_jacobian_parity(name, op, cfgs, knobs):
    """Exact derivative within TOL_EXACT; for the PNP operator also the compact 5-plane export (matrix_compact)."""
    c, m, p = make_ctx(name, cfgs[1])
    u, a0, a1 = _state(m, op, 3)
    _, _, val_o, ab = ora.jacobian(m, p, op, u, a0, a1, valency=-1.0, mode=1, want_abs=True)
    for compact in ((0, 1) if op == ora.OP_PNP else (0,)):
        knobs(matrix_compact=compact)
        val = _jacobian(c, m, op, 1)[4]
        err = rel_err(val, val_o, ab)
        print("FIGURE exact_jacobian %s op=%d compact=%d max_rel=%.3g" % (name, op, compact, err))
        assert err <= TOL_EXACT


# ---------------------------------------------------------------------------------------------------------------------
# SpMV
SPMV_SETTINGS = [dict(tma=0), dict(tma=1, tma_min_rows=1, tma_lpr=1), dict(tma=1, tma_min_rows=1, tma_lpr=2)]


@pytest.mark.parametrize("planes", [1, 5, 7])
@pytest.mark.parametrize("name", ALL)
def test_spmv_within_the_exact_sum_bound(name, planes, cfgs, knobs):
    """y = A x of an exact Jacobian (PB: 1 plane; PNP: 5 or 7) against the correctly rounded sum of each exported row:
    |y - y_ref| <= gamma(n) sum|a_ij x_j| + u |y_ref|, n = the row's terms.  Plain-load kernel and streaming kernel with
    1 and 2 lanes per row.  Dot and norm of the product against the reference within 1e-12."""
    capi = _capi()
    op = ora.OP_PB if planes == 1 else ora.OP_PNP
    F = ora.nfields(op)
    c, m, _ = make_ctx(name, cfgs[1])
    knobs(matrix_compact=1 if planes == 5 else 0)
    _, A, rp, col, val, _ = _jacobian(c, m, op, capi.JAC_ANALYTIC, seed=7)
    x = np.random.RandomState(11).uniform(-1, 1, F * m.nv)
    p, e = two_prod(val, x[col])
    y_ref = np.array([math.fsum(np.concatenate([p[i:j], e[i:j]])) for i, j in zip(rp[:-1], rp[1:])])
    S = np.add.reduceat(np.abs(p), rp[:-1])
    bound = gamma(np.diff(rp)) * S + U * np.abs(y_ref)
    vx, vy = c.vec(F, x), c.vec(F)
    for kw in SPMV_SETTINGS:
        knobs(**kw)
        c.vec_set(vy, np.nan)
        c.spmv(A, vx, vy)
        y = c.download(vy, F)
        print("FIGURE spmv %s planes=%d %s max_excess=%.3g" % (name, planes, kw, np.max(np.abs(y - y_ref) / np.maximum(bound, 1e-300))))
        assert np.all(np.abs(y - y_ref) <= bound), (kw, np.max(np.abs(y - y_ref) - bound))
        assert abs(c.dot(vx, vy) - x @ y_ref) <= 1e-12 * (np.abs(x) @ S)
        assert abs(c.norm(vy) - np.linalg.norm(y_ref)) <= 1e-12 * np.linalg.norm(y_ref)


# ---------------------------------------------------------------------------------------------------------------------
# solvers
@pytest.mark.parametrize("prec,steps", [(2, 1), (2, 3), (3, 1)])
@pytest.mark.parametrize("op", [ora.OP_PB, ora.OP_PNP])
@pytest.mark.parametrize("name", ALL)
def test_ssor_ilu0_application_equals_sequential_sweep(name, op, prec, steps, cfgs):
    """SSOR(1), SSOR(3), ILU0: the level-scheduled sweep equals the oracle's sequential one; the hub couples a long chain
    of dofs into the level schedule.  Bar: 1e-12 relative, as on the shipped meshes, or -- where the application itself
    is that sensitive to rounding -- 10 times the largest change of the oracle's result under random relative
    perturbations of 1 u of the matrix and right-hand side (ILU0 of the PNP matrix with a 600-slot hub row: up to 1e-10;
    an error in the schedule changes the result by O(1))."""
    capi = _capi()
    c, m, _ = make_ctx(name, cfgs[1])
    F = ora.nfields(op)
    _, A, rp, col, val, _ = _jacobian(c, m, op, capi.JAC_ANALYTIC, seed=7)
    d = np.random.RandomState(5).uniform(-1, 1, F * m.nv)
    s = c.solver(capi.SOLVER_BCGS, prec, 100, steps)
    vv = c.vec(F)
    c.precond_apply(s, A, c.vec(F, d), vv)
    v_o = ora.prec_apply(rp, col, val, d, prec, steps)
    spread = 0.0
    for k in range(3):
        rng = np.random.RandomState(20 + k)
        v_p = ora.prec_apply(rp, col, val * (1 + U * rng.uniform(-1, 1, len(val))), d * (1 + U * rng.uniform(-1, 1, len(d))),
                             prec, steps)
        spread = max(spread, np.linalg.norm(v_p - v_o))
    err = np.linalg.norm(c.download(vv, F) - v_o)
    print("FIGURE sweep %s op=%d prec=%d steps=%d rel=%.3g perturbation_rel=%.3g"
          % (name, op, prec, steps, err / np.linalg.norm(v_o), spread / np.linalg.norm(v_o)))
    assert err <= max(1e-12 * np.linalg.norm(v_o), 10 * spread)


@pytest.mark.parametrize("compact", [0, 1])
def test_multigrid_bicgstab_on_the_refined_hub(compact, cfgs, knobs):
    """BiCGSTAB + multigrid (geometric levels, re-discretised coarse operators: the hub's 600-slot row puts a chunk of every
    level above JAC_CAP) on the PNP Jacobian of the twice-refined hub mesh, 7 planes and compact: converges, and the true
    residual of the exported matrix is within twice the requested reduction.  The thin elements around the hub make the
    point-block smoother weak: close to 300 iterations."""
    capi = _capi()
    knobs(matrix_compact=compact)
    c, m, p = make_ctx("hub600_ref2", cfgs[1])
    h = c.operator(capi.OP_PNP, 0)
    u = c.vec(3); c.vec_set(u, 0.05)
    A = c.matrix(h)
    c.jacobian(h, u, A, capi.JAC_ANALYTIC, 0.0)
    b = np.random.RandomState(0).uniform(-1, 1, 3 * m.nv)
    b[c.constraints(h, 3)] = 0.0
    s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 3000, 2)
    z, r = c.vec(3), c.vec(3, b)
    res = c.solve(s, A, z, r, 1e-8)
    assert res.converged
    rp, col = c.pattern(h, 3)
    val = c.matrix_values(h, A, len(col))
    print("FIGURE multigrid compact=%d iterations=%d" % (compact, res.iterations))
    assert np.linalg.norm(b - ora.spmv(rp, col, val, c.download(z, 3))) <= 2e-8 * np.linalg.norm(b)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name", BASE)
def test_newton_pb_matches_oracle(name, mode, cfgs):
    """PB Newton with BiCGSTAB + Jacobi: the oracle's iteration count, and the device's field solves the oracle's problem
    to 10x the cfg's reduction of the oracle's first defect.  (The two fields differ by up to 1e-5 relative: the thin
    elements make the system ill-conditioned, and a defect reduction of 1e-8 fixes the field only to that.)"""
    capi = _capi()
    c, m, p = make_ctx(name, cfgs[1])
    h = c.operator(capi.OP_PB, 0)
    vu = c.vec(1)
    st, res = c.newton(h, vu, c.solver(capi.SOLVER_BCGS, capi.PREC_JACOBI, 5000), c.newton_opts(jac_mode=mode))
    opts = ora.newton_opts(p, solver=ora.SOLVER_BCGS, prec=ora.PREC_JACOBI, jac_mode=mode)
    opts[12] = 5000
    u_o, res_o = ora.newton(m, p, ora.OP_PB, np.zeros(m.nv), opts)
    assert res.converged and res_o["converged"]
    assert res.iterations == res_o["iterations"]
    r = ora.residual(m, p, ora.OP_PB, c.download(vu, 1))
    assert np.linalg.norm(r) <= 10 * p.sys[7] * res_o["first_defect"]


# ---------------------------------------------------------------------------------------------------------------------
# outputs
@pytest.mark.parametrize("name", ALL)
def test_interpolate_bcext_and_ion_flux(name, cfgs):
    """interpolate_bcext (precedence at vertices of two surfaces) and calcIonFlux, whose surface normals follow the
    segments' direction (reversed segments).  Constrained values that are a surface's Dirichlet constant are exact.  (At
    some Dirichlet-Neumann junctions the reference's BCExtension takes the Neumann surface and returns c0 exp(-+pb) for a
    constrained dof; there the device's exp and the host's may differ in the last bit.)"""
    c, m, p = make_ctx(name, cfgs[1])
    pb = np.random.RandomState(4).uniform(-1, 1, m.nv)
    vpb, vout = c.vec(1, pb), c.vec(1)
    for comp in range(3):
        c.interpolate_bcext(comp, vpb, vout)
        got, want = c.download(vout, 1), ora.interpolate(m, p, comp, pb)
        assert np.max(np.abs(got - want)) <= 1e-14 * max(1.0, np.max(np.abs(want)))
        d = ora.dirichlet(m, p, 1, comp) & np.isin(want, p.surf[p.surf[:, 3 * comp] == 0, 3 * comp + 2])
        assert d.any() and np.array_equal(got[d], want[d])
    rng = np.random.RandomState(5)
    phi = 0.4 * np.sin(0.2 * m.x) + 0.1 * m.y
    cp = 0.06 * np.exp(-phi) * (1 + 0.05 * rng.uniform(-1, 1, m.nv)); cm = 0.06 * np.exp(phi) * (1 + 0.05 * rng.uniform(-1, 1, m.nv))
    ip, im = c.ion_flux(c.vec(1, phi), c.vec(1, cp), c.vec(1, cm))
    ip_o, im_o = ora.ion_flux(m, p, phi, cp, cm)
    ip_a, im_a = ora.ion_flux(m, p, np.abs(phi), np.abs(cp), np.abs(cm))
    scale = np.abs(ip_o).max() + np.abs(im_o).max() + np.abs(ip_a).max() + np.abs(im_a).max()
    assert np.all(np.abs(ip - ip_o) <= 1e-11 * scale) and np.all(np.abs(im - im_o) <= 1e-11 * scale)
    assert np.any(ip_o != 0)


# ---------------------------------------------------------------------------------------------------------------------
# quadratic and cubic elements
P_MESH = "hub16_open"   # mixed orientation in every ring, reversed segments, the hub on the boundary


@pytest.mark.parametrize("degree", [2, 3])
def test_pk_pattern_and_constraints_bit_exact(degree, cfgs):
    capi = _capi()
    c, m, p = make_ctx(P_MESH, cfgs[1], degree=degree)
    P = ora.P2(m, p, degree)
    va, vb = c.space_edges()
    assert np.array_equal(va, P.eva) and np.array_equal(vb, P.evb)
    for op, F, comp0 in ((capi.OP_PB, 1, 0), (capi.OP_DIFFUSION, 1, 1), (capi.OP_MASS, 1, 2), (capi.OP_PNP, 3, 0)):
        h = c.operator(op, comp0)
        assert np.array_equal(c.constraints(h, F), P.dirichlet(F, comp0))
        rp, col = c.pattern(h, F)
        rp_o, col_o = P.pattern(F, comp0)
        assert np.array_equal(rp, rp_o) and np.array_equal(col, col_o)


@pytest.mark.parametrize("degree,intorder", DEG_ORDER)
@pytest.mark.parametrize("op", OPS)
def test_pk_residual_and_jacobians(op, degree, intorder, cfgs):
    """residual within TOL, FD Jacobian within TOL, exact derivative within TOL_EXACT (test_gpu_p2's bars)"""
    c, m, p = make_ctx(P_MESH, cfgs[1], degree=degree)
    P = ora.P2(m, p, degree)
    F = ora.nfields(op)
    rng = np.random.RandomState(0)
    u, a0, a1 = rng.uniform(-1, 1, F * P.nd), rng.uniform(0, 1, P.nd), rng.uniform(0, 1, P.nd)
    h = _operator(c, op, a0, a1)
    if intorder:
        c.operator_set_intorder(h, intorder)
    vu, vr = c.vec(F, u), c.vec(F)
    c.residual(h, vu, vr)
    r_o, ab = P.residual(op, u, a0, a1, valency=-1.0, want_abs=True, intorder=intorder or -1)
    assert rel_err(c.download(vr, F), r_o, ab) <= TOL
    for mode in (0, 1):
        A = c.matrix(h)
        c.jacobian(h, vu, A, mode, 1e-11)
        rp, col, val_o, ab = P.jacobian(op, u, a0, a1, valency=-1.0, mode=mode, eps=1e-11, want_abs=True, intorder=intorder or -1)
        err = rel_err(c.matrix_values(h, A, len(col)), val_o, ab)
        print("FIGURE pk degree=%d intorder=%d op=%d mode=%d max_rel=%.3g" % (degree, intorder, op, mode, err))
        assert err <= (TOL if mode == 0 else TOL_EXACT)
