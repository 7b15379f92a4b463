"""GPU tests of the multigrid's single-precision companion planes (pnp_amg.cu, mg_f32_rule; pnp_tune "mg_f32_min_rows"):
on a level that has one, the first Jacobi sweep, every damped point-block Jacobi step and the residual apply the level's
matrix rounded to float32 planes and widened to double, while the Krylov method keeps applying the fp64 matrix.

  * one smoother step / residual is exactly damped block-Jacobi on A32 = fl32(A), within the rounding bound of
    test_gpu_compact_layout's numpy restatement, and not the fp64 result;
  * a solve to 1e-13 under the forced rule satisfies the oracle's system as tightly as the fp64 preconditioner does;
  * one Newton step at the default rule takes the iterations and line-search trials of the fp64 preconditioner, and each
    update meets the step's own stopping criterion against the fp64 Jacobian;
  * bytes: fine-level residual and smoother launches read 4 bytes less per plane and slot, nothing else changes;
  * scope: Chebyshev, Gauss-Seidel, the plain-load kernel and partitioned hierarchies read what they read without it.
"""
import numpy as np
import pytest
import scipy.sparse as sp

import util
from oracle import binding as ora
from test_gpu_compact_layout import (assembled, block_inverse, diag_blocks, entry_fields, export, gamma, make_ctx,
                                     newton_state, smooth_state, smoother_reference)
from test_gpu_parity import TOL_EXACT

pytestmark = pytest.mark.gpu

OFF = 1e30  # mg_f32_min_rows above any level: no companion
DEFAULT_TUNE = dict(mg_f32_min_rows=-1, tma=1, tma_min_rows=-1, tma_lpr=2, tma_stages=2, matrix_compact=0, jac_compact=1)


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


def rounded_planes(rp, col, val, nv, planes):
    """the exported matrix with every value PLANE rounded to float32 (the companion), entries recomputed in double as
    pnp_block() does.  7 planes: each entry is a plane.  5 planes: L, M, P, Q are entries; the (c+,c+) and (c-,c-)
    entries are L - D and L + D, so D is recovered as their half difference (exact where no rounding intervened, within
    an fp64 ulp of L + D else, which moves fl32(D) only where D lies that close to a float32 rounding boundary)."""
    r = val.astype(np.float32).astype(np.float64)
    if planes == 7:
        return r
    row, ki, kj = entry_fields(rp, col, nv)
    b00, b11, b22 = ((ki == k) & (kj == k) for k in range(3))
    L = val[b00]
    D = (val[b22] - val[b11]) / 2
    L32, D32 = L.astype(np.float32).astype(np.float64), D.astype(np.float32).astype(np.float64)
    r[b11] = L32 - D32
    r[b22] = L32 + D32
    return r


def smoother_case(c, h, A, nv, planes, nu):
    capi = _capi()
    rp, col, val = export(c, h, A)
    b = np.random.RandomState(9).uniform(-1, 1, 3 * nv)
    vb, vy = c.vec(3, b), c.vec(3)
    s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 1, 1)
    for k, v in (("amg_smoother", 0), ("amg_pre_steps", nu), ("amg_post_steps", 0), ("amg_alpha", 0.0),
                 ("amg_dense_max", 0), ("amg_geometric", 0), ("amg_coarse_sweeps", 0)):
        c.solver_set_option(s, k, v)
    c.precond_apply(s, A, vb, vy)
    y = c.download(vy, 3)
    out = {}
    for name, v in (("f32", rounded_planes(rp, col, val, nv, planes)), ("f64", val)):
        As = sp.csr_matrix((v, col, rp), shape=(3 * nv, 3 * nv))
        Dinv, E, _, _ = block_inverse(diag_blocks(rp, col, v, nv))
        out[name] = smoother_reference(As, Dinv, E, b, nu, 0)
    return y, out


@pytest.mark.parametrize("name", ["pore_without_dna", "fan"])
@pytest.mark.parametrize("planes", [5, 7])
@pytest.mark.parametrize("lpr", [1, 2])
def test_smoother_step_is_damped_jacobi_on_the_rounded_matrix(name, planes, lpr, knobs):
    """nu = 1, 2, 3 pre-smoothing steps on the fine level alone (no coarse correction, as in test_gpu_compact_layout's
    test_one_smoother_step_matches_numpy) with the companion forced on every level (mg_f32_min_rows = 1, streaming kernel
    everywhere): the result is the numpy recurrence on fl32(A) within twice its rounding bound, and NOT the fp64 one.
    nu = 1 is the stored block inverses (k_dinv of the rounded blocks), nu >= 2 the streaming kernel's smoother; "fan"
    has an over-full first tile, whose slots the kernel reads from the float planes in global memory."""
    capi = _capi()
    c, _, _ = make_ctx(name, 0, oracle=False)
    g = c.mesh_get()
    nv = len(g["x"])
    h = c.operator(capi.OP_PNP, 0)
    A = assembled(c, h, newton_state(g["x"], g["y"]), planes == 5, knobs)
    knobs(mg_f32_min_rows=1, tma_min_rows=1, tma_lpr=lpr)
    for nu in (1, 2, 3):
        y, ref = smoother_case(c, h, A, nv, planes, nu)
        x, dx = ref["f32"]
        assert np.all(np.abs(y - x) <= 2 * dx), (nu, np.max(np.abs(y - x) - 2 * dx))
        x64, dx64 = ref["f64"]
        assert not np.all(np.abs(y - x64) <= 2 * dx64), nu


def oracle_solve_bound(c, m, p, h, u0, solver, red):
    """test_workspace_reads_five_planes_and_solves_the_oracle_system's check of the step z of slp at reduction `red`"""
    capi = _capi()
    vu = c.vec(3, u0)
    res = c.slp(h, vu, solver, red, jac_mode=capi.JAC_ANALYTIC, eps=0.0)
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
    return res


@pytest.mark.parametrize("name", ["pore", "one_wall"])
def test_forced_rule_solves_the_oracle_system(name, knobs):
    """slp with the multigrid (meshes refined once, companion on every level) at reduction 1e-13: the accuracy the solve
    reaches is the Krylov operator's, which stays fp64"""
    capi = _capi()
    c, m, p = make_ctx(name, 1)
    knobs(mg_f32_min_rows=1, tma_min_rows=1)
    oracle_solve_bound(c, m, p, c.operator(capi.OP_PNP, 0), smooth_state(m.x, m.y),
                       c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 20000, 1), 1e-13)


def step_linear_residual(c, h, us, u):
    """||J(u_s) (u_s - u) - F(u_s)|| / ||F(u_s)||: the fp64 linear residual of a Newton step's update (u = u_s - z with
    J z = F, pnp_newton.cu), J the exact Jacobian in a 7-plane user matrix"""
    capi = _capi()
    A = c.matrix(h)
    c.jacobian(h, us, A, capi.JAC_ANALYTIC, 0.0)
    d, y, r = c.vec(3), c.vec(3), c.vec(3)
    c.vec_copy(d, us); c.axpy(d, -1.0, u)
    c.spmv(A, d, y)
    c.residual(h, us, r)
    c.axpy(y, -1.0, r)
    out = c.norm(y) / c.norm(r)
    for v in (d, y, r):
        c.vec_destroy(v)
    c.matrix_destroy(A)
    return out


def newton_step_both_rules(levels, rules):
    """bench.py's state (nested iteration from level 3) on pore refined `levels` times, one Newton step per rule"""
    import bench
    capi = _capi()
    c = capi.Context(0)
    a, cfg = bench.load_case()
    c.mesh_set(**a); c.params_read(cfg)
    h, s, us = bench.build_state(c, capi, levels, 3, capi.JAC_ANALYTIC, 2, False)
    opts = c.newton_opts(jac_mode=capi.JAC_ANALYTIC, max_iterations=1)
    u = c.vec(3)
    out = {}
    for rule in rules:
        capi.tune("mg_f32_min_rows", rule)
        c.vec_copy(u, us)
        c.profile_bytes(reset=True)
        st, r = c.newton(h, u, s, opts, check=False)
        assert st in (0, 1), st
        fine = c.profile_bytes(reset=True)["spmv_fine"]
        out[rule] = dict(its=r.linear_iterations, trials=r.line_search_trials, fine=fine,
                         lin_res=step_linear_residual(c, h, us, u))
    return out, opts.min_linear_reduction


def test_newton_step_iterations_at_the_default_rule(knobs):
    """pore refined 6 times (11.8 M vertices: the default rule puts the top level on the companion): the same linear
    iterations and line-search trials as without it, and each update meets the step's stopping criterion against the
    fp64 Jacobian, ||J d - F|| <= min_linear_reduction ||F||"""
    out, mlr = newton_step_both_rules(6, (-1, OFF))
    assert out[-1]["fine"] < out[OFF]["fine"]  # the default rule did pick the top level
    assert out[-1]["its"] == out[OFF]["its"] and out[-1]["trials"] == out[OFF]["trials"], out
    for rule in out:
        assert out[rule]["lin_res"] <= mlr, (rule, out[rule])


def slp_profile(c, h, u0, solver_opts, rule, knobs, planes=5):
    capi = _capi()
    knobs(mg_f32_min_rows=rule, jac_compact=1 if planes == 5 else 0)
    s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 2, 1)
    for k, v in solver_opts.items():
        c.solver_set_option(s, k, v)
    c.profile_spmv(True)
    c.profile_bytes(reset=True)
    c.slp(h, c.vec(3, u0), s, 1e-30, jac_mode=capi.JAC_ANALYTIC, eps=0.0)
    launches = c.profile_spmv_get()[0]
    c.profile_spmv(False)
    return c.profile_bytes(reset=True), launches


@pytest.mark.parametrize("planes", [5, 7])
def test_companion_bytes(planes, knobs):
    """two BiCGSTAB iterations of the linear-problem step on pore refined once, rule forced against off: the same fine-level
    launches of every kind, and fine-level SpMV bytes lower by exactly 4 P ns per residual and smoother launch"""
    capi = _capi()
    c, _, _ = make_ctx("pore", 1, oracle=False)
    g = c.mesh_get()
    ns = c.mesh_sizes()["nslots"]
    h = c.operator(capi.OP_PNP, 0)
    knobs(tma_min_rows=1)
    u0 = smooth_state(g["x"], g["y"])
    b_on, l_on = slp_profile(c, h, u0, {}, 1, knobs, planes)
    b_off, l_off = slp_profile(c, h, u0, {}, OFF, knobs, planes)
    assert l_on == l_off and l_on[1] > 0 and l_on[2] > 0, (l_on, l_off)
    assert b_off["spmv_fine"] - b_on["spmv_fine"] == 4.0 * planes * ns * (l_on[1] + l_on[2]), (b_on, b_off, l_on)


@pytest.mark.parametrize("case", ["chebyshev", "gauss_seidel", "plain_kernel"])
def test_no_companion_outside_the_rule(case, knobs):
    """Chebyshev, Gauss-Seidel (7 planes) and tma = 0: forcing the rule reads the same bytes as switching it off"""
    capi = _capi()
    c, _, _ = make_ctx("pore", 1, oracle=False)
    g = c.mesh_get()
    h = c.operator(capi.OP_PNP, 0)
    knobs(tma_min_rows=1, tma=0 if case == "plain_kernel" else 1)
    opts = {"chebyshev": {"amg_smoother": 1}, "gauss_seidel": {"amg_smoother": 2}, "plain_kernel": {}}[case]
    u0 = smooth_state(g["x"], g["y"])
    on = slp_profile(c, h, u0, opts, 1, knobs)
    off = slp_profile(c, h, u0, opts, OFF, knobs)
    assert on == off and on[0]["spmv_fine"] > 0, (on, off)


def test_no_companion_on_partitioned_hierarchies(knobs):
    """the distributed multigrid with a replicated coarsest level (one subdomain, as in test_gpu_partitioned): forcing the
    rule reads the same bytes on every level as switching it off"""
    capi = _capi()
    from dune_pnp_b200 import partition
    a = util.load_mesh_arrays("pore")
    plans = partition.build_hierarchy(a, 1, 0, 2)
    root = capi.Context(0)
    children = partition.setup_distributed(capi, root, plans, util.cfg_path("pore"), 0, 1, None, replica_mesh=a, replica_level=0)
    h = root.operator(capi.OP_PNP, 0)
    nv = root.mesh_sizes()["nv"]
    knobs(tma_min_rows=1)
    b = np.random.RandomState(0).uniform(-1, 1, 3 * nv)
    b[root.constraints(h, 3)] = 0.0
    out = []
    for rule in (1, OFF):
        knobs(mg_f32_min_rows=rule)
        u = root.vec(3); root.vec_set(u, 0.05)
        A = root.matrix(h)
        root.jacobian(h, u, A, capi.JAC_ANALYTIC, 0.0)
        s = root.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 200, 2)
        z, r = root.vec(3), root.vec(3, b)
        root.profile_bytes(reset=True)
        res = root.solve(s, A, z, r, 1e-8)
        assert res.converged
        out.append((res.iterations, root.profile_bytes(reset=True)))
    assert out[0] == out[1], out
    del children
    root.close()
