"""GPU parity on the HEADLINE configuration's own mesh (test/pore_pnp: pore.msh + pore.cfg) and at sizes where the
locality renumbering, the staged Jacobian tiles and the multi-pass SpMV rows are all exercised:

  * the reference flow `stationary_pnp_from_pb` (stationary_pnp_from_pb.hh:92-370 with test/pore_pnp/pore.cfg:7-12) on
    the pore mesh, refinement levels 0 and 1, against the oracle run of the same flow (equal Newton iteration counts,
    fields within 1e-8 relative L2) and against the committed golden solution (tests/golden/pore_solution.npz);
  * residual, both Jacobian flavours and SpMV against the oracle on refinement level 4 (738 k vertices, 2.2 M dofs) and
    residual / exact Jacobian / SpMV on level 5 (2.9 M vertices, 8.8 M dofs).
"""
import os

import numpy as np
import pytest

import util
from oracle import binding as ora
from test_gpu_parity import TOL, TOL_EXACT, _capi, make_ctx, rel_err

pytestmark = pytest.mark.gpu


def _pnp_from_pb_gpu(c, tight, prec_steps=2, jac_mode=None):
    """PB Newton -> interpolate(BCExtension) -> PNP Newton on the device (multigrid-preconditioned BiCGSTAB).  tight: both
    sides use the exact-derivative Jacobian (with the forward differences' noise of ~1e-5 in the entries, whether a run to
    1e-11 needs one Newton step more or less is a coin toss)."""
    capi = _capi()
    kw = dict(reduction=1e-11, min_linear_reduction=1e-9, jac_mode=capi.JAC_ANALYTIC if jac_mode is None else jac_mode) if tight else {}
    hpb = c.operator(capi.OP_PB, 0)
    vpb = c.vec(1)
    st, rpb = c.newton(hpb, vpb, c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 20000, prec_steps), c.newton_opts(**kw))
    f = [c.vec(1) for _ in range(3)]
    for k in range(3):
        c.interpolate_bcext(k, vpb, f[k])
    vu = c.vec(3)
    c.pack3(vu, *f)
    u0 = c.download(vu, 3)
    h = c.operator(capi.OP_PNP, 0)
    st, res = c.newton(h, vu, c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 20000, prec_steps), c.newton_opts(**kw))
    return c.download(vpb, 1), rpb, u0, c.download(vu, 3), res


def _pnp_from_pb_oracle(m, p, tight):
    """The same flow in the oracle; ILU0-preconditioned BiCGSTAB keeps the CPU side to seconds (the Newton path only
    needs linear solves of the requested accuracy, SURVEY H3)."""
    opts = ora.newton_opts(p, solver=ora.SOLVER_BCGS, prec=ora.PREC_ILU0, jac_mode=1 if tight else 0); opts[12] = 20000
    if tight:
        opts[0], opts[2] = 1e-11, 1e-9
    pb, rpb = ora.newton(m, p, ora.OP_PB, np.zeros(m.nv), opts)
    u0 = np.concatenate([ora.interpolate(m, p, k, pb) for k in range(3)])
    u, r = ora.newton(m, p, ora.OP_PNP, u0, opts)
    return pb, rpb, u0, u, r


@pytest.mark.parametrize("levels,tight", [(0, False), (0, True), (1, False), (1, True), (2, True)])
def test_stationary_pnp_from_pb_on_pore_matches_oracle(levels, tight):
    """tight=False: pore.cfg's own Newton settings (reduction 1e-9 / linear reduction 1e-8, test/pore_pnp/pore.cfg:7-12):
    equal Newton iteration counts; two runs that both stop at that reduction agree to about 10x the reduction in the
    defect, i.e. ~1e-8 .. 1e-7 in the fields (measured 1.6e-8).  tight=True (1e-11 / 1e-9): CONVERGED fields, within 1e-8."""
    c, m, p = make_ctx("pore", levels=levels)
    pb, rpb, u0, u, res = _pnp_from_pb_gpu(c, tight=tight)
    pb_o, rpb_o, u0_o, u_o, res_o = _pnp_from_pb_oracle(m, p, tight=tight)
    assert rpb.converged and rpb_o["converged"] and rpb.iterations == rpb_o["iterations"]
    assert np.linalg.norm(pb - pb_o) <= 1e-8 * np.linalg.norm(pb_o)
    assert np.linalg.norm(u0 - u0_o) <= 1e-8 * np.linalg.norm(u0_o)
    assert res.converged and res_o["converged"]
    assert res.iterations == res_o["iterations"]
    nv = m.nv
    tol = 1e-8 if tight else 1e-7
    for k in range(3):
        assert np.linalg.norm(u[k * nv:(k + 1) * nv] - u_o[k * nv:(k + 1) * nv]) <= tol * np.linalg.norm(u_o[k * nv:(k + 1) * nv])
    # defect histories of the two Newton runs agree as far as the linear solves' accuracy lets them
    assert abs(res.first_defect - res_o["first_defect"]) <= 1e-7 * res_o["first_defect"]


def test_pore_golden_solution():
    """tests/golden/pore_solution.npz (scripts/make_golden_solutions.py: BiCGSTAB + SSOR(1), FD Jacobian, reduction 1e-11):
    the device run with its own solver stack (multigrid-preconditioned BiCGSTAB) and the same FD Jacobian lands on the same
    fields in the same number of Newton steps."""
    capi = _capi()
    z = np.load(os.path.join(util.GOLDEN, "pore_solution.npz"))
    c, m, p = make_ctx("pore")
    pb, rpb, u0, u, res = _pnp_from_pb_gpu(c, tight=True, jac_mode=capi.JAC_FD_FAITHFUL)
    assert rpb.iterations == int(z["pb_newton_iterations"]) and res.iterations == int(z["pnp_newton_iterations"])
    assert np.linalg.norm(pb - z["pb"]) <= 1e-8 * np.linalg.norm(z["pb"])
    assert np.linalg.norm(u0 - z["u0"]) <= 1e-8 * np.linalg.norm(z["u0"])
    nv = m.nv
    for k in range(3):
        assert np.linalg.norm(u[k * nv:(k + 1) * nv] - z["u"][k * nv:(k + 1) * nv]) <= 1e-8 * np.linalg.norm(z["u"][k * nv:(k + 1) * nv])
    # and with the reference's own jacobian_volume (FD-faithful) through the reference's default backend's cousin ILU0
    c2, _, _ = make_ctx("pore")
    h = c2.operator(capi.OP_PNP, 0)
    vu = c2.vec(3, z["u0"])
    st, r2 = c2.newton(h, vu, c2.solver(capi.SOLVER_BCGS, capi.PREC_ILU0, 20000, 1),
                       c2.newton_opts(jac_mode=capi.JAC_FD_FAITHFUL, reduction=1e-11, min_linear_reduction=1e-9))
    assert r2.converged and r2.iterations == int(z["pnp_newton_iterations"])
    assert np.linalg.norm(c2.download(vu, 3) - z["u"]) <= 1e-8 * np.linalg.norm(z["u"])
    d = z["pnp_defects"]
    assert abs(r2.first_defect - d[0]) <= 1e-10 * d[0]


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """`bench.py --dump-outputs` at k = 4 (2.2 M dofs): the last timed Newton step's state and result are written, and a
    second run with the same arguments writes the same bits (the start state and the step are deterministic), so that two
    builds can be compared output for output."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lines = {}
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--levels", "4", "--steps", "2", "--warmup", "1",
                              "--no-cpu", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
        lines[run] = json.loads(out.stdout.strip().splitlines()[-1])
    u, res = np.load(tmp_path / "a" / "u.npy"), np.load(tmp_path / "a" / "newton_result.npy")
    assert u.dtype == np.float64 and u.shape == (3, 738033) and np.all(np.isfinite(u))
    assert res.dtype == np.float64 and res[1] == 1 and res[3] == lines["a"]["defect_after"] and res[3] < res[2]
    for name in ("u.npy", "newton_result.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)), name


def _smooth_state(m, op):
    """A smooth, physically shaped state (potential O(1), concentrations around c0) plus deterministic noise."""
    rng = np.random.RandomState(21)
    phi = 0.8 * np.sin(0.07 * m.x) * np.cos(0.05 * m.y) + 0.05 * rng.uniform(-1, 1, m.nv)
    if ora.nfields(op) == 1:
        return phi
    return np.concatenate([phi, 0.06 * np.exp(-phi) * (1 + 0.02 * rng.uniform(-1, 1, m.nv)),
                           0.06 * np.exp(phi) * (1 + 0.02 * rng.uniform(-1, 1, m.nv))])


@pytest.mark.parametrize("op", [ora.OP_PB, ora.OP_PNP])
def test_kernel_parity_level4(op):
    """738 033 vertices: every residual entry and every entry of both Jacobians within 1e-12 of the oracle's (relative to
    the entry's absolute element contributions, see module docstring of test_gpu_parity), SpMV likewise."""
    capi = _capi()
    c, m, p = make_ctx("pore", levels=4)
    assert m.nv == 738033
    F = ora.nfields(op)
    u = _smooth_state(m, op)
    h = c.operator(op, 0)
    vu, vr, A = c.vec(F, u), c.vec(F), c.matrix(h)
    c.residual(h, vu, vr)
    r_o, ab = ora.residual(m, p, op, u, want_abs=True)
    assert rel_err(c.download(vr, F), r_o, ab) <= TOL
    rp_g, col_g = c.pattern(h, F)
    val = None
    for mode in (0, 1):
        c.jacobian(h, vu, A, mode, 1e-11)
        rp, col, val_o, jab = ora.jacobian(m, p, op, u, mode=mode, eps=1e-11, want_abs=True)
        assert np.array_equal(rp, rp_g) and np.array_equal(col, col_g)
        val = c.matrix_values(h, A, len(col))
        assert rel_err(val, val_o, jab) <= (TOL if mode == 0 else TOL_EXACT)
        if mode == 0:
            assert np.mean(val == val_o) > 0.9   # two-term sums reproduce the oracle bit for bit
    x = np.random.RandomState(5).uniform(-1, 1, F * m.nv)
    vx, vy = c.vec(F, x), c.vec(F)
    c.spmv(A, vx, vy)
    y_o = ora.spmv(rp_g, col_g, val, x)
    scale = ora.spmv(rp_g, col_g, np.abs(val), np.abs(x))
    assert rel_err(c.download(vy, F), y_o, scale) <= TOL
    assert abs(c.norm(vy) - np.linalg.norm(y_o)) <= 1e-12 * np.linalg.norm(y_o)


def test_residual_jacobian_spmv_parity_level5():
    """2 946 529 vertices (k = 5, the CPU baseline's size): PNP residual, scalar PB Jacobian (exact derivative) and the
    SpMV with it against the oracle."""
    capi = _capi()
    c, m, p = make_ctx("pore", levels=5)
    assert m.nv == 2946529
    u3 = _smooth_state(m, ora.OP_PNP)
    h3 = c.operator(capi.OP_PNP, 0)
    vu, vr = c.vec(3, u3), c.vec(3)
    c.residual(h3, vu, vr)
    r_o, ab = ora.residual(m, p, ora.OP_PNP, u3, want_abs=True)
    assert rel_err(c.download(vr, 3), r_o, ab) <= TOL
    u1 = u3[:m.nv]
    h1 = c.operator(capi.OP_PB, 0)
    v1, A = c.vec(1, u1), c.matrix(h1)
    c.jacobian(h1, v1, A, capi.JAC_ANALYTIC, 0.0)
    rp, col, val_o, jab = ora.jacobian(m, p, ora.OP_PB, u1, mode=1, want_abs=True)
    val = c.matrix_values(h1, A, len(col))
    assert rel_err(val, val_o, jab) <= TOL_EXACT
    x = np.cos(0.11 * m.x + 0.3) * np.sin(0.13 * m.y)
    vx, vy = c.vec(1, x), c.vec(1)
    c.spmv(A, vx, vy)
    y_o = ora.spmv(rp, col, val, x)
    assert rel_err(c.download(vy, 1), y_o, ora.spmv(rp, col, np.abs(val), np.abs(x))) <= TOL


@pytest.fixture
def streaming_everywhere():
    capi = _capi()
    capi.tune("tma_min_rows", 1)
    yield
    capi.tune("tma_min_rows", -1)


def test_streaming_spmv_kernel_on_the_small_meshes(streaming_everywhere):
    """k_star_op_tma (bulk-copy pipeline, pnp_spmv_tma.cuh) normally serves levels with >= 2 tiles per SM; with the tuning
    knob tma_min_rows = 1 every SpMV / multigrid level operation of these small-mesh parity tests goes through it: partial
    last tiles, tiles of unrefined Gmsh meshes with more slots than a stage holds (plain-load fallback), gather windows
    clipped at both ends, both plane counts."""
    import test_gpu_parity as t
    for name, levels in (("sphere", 0), ("pore", 0), ("pore_small", 2), ("cylinder", 1)):
        for op in (ora.OP_PB, ora.OP_PNP):
            t.test_spmv_parity(name, levels, op)
    for kind, prec in ((0, 0), (0, 1), (1, 0), (1, 1)):
        t.test_linear_solvers_on_poisson(kind, prec)
    for op in (ora.OP_PB, ora.OP_PNP):
        for geometric in (0, 1):
            t.test_multigrid_preconditioner(op, geometric)
    t.test_multigrid_options(0, 2)
    t.test_newton_pnp_from_pb_matches_oracle("pore_small", False)


def test_streaming_and_plain_spmv_agree_level4(streaming_everywhere):
    """The two SpMV kernels on the same 738 k-vertex matrix: all three epilogues of the multigrid cycle, compared through
    one V(2,2) application (identical arithmetic per row up to the summation order inside a row)."""
    capi = _capi()
    c, m, p = make_ctx("pore", levels=4)
    h = c.operator(capi.OP_PNP, 0)
    u = c.vec(3, _smooth_state(m, ora.OP_PNP))
    A = c.matrix(h)
    c.jacobian(h, u, A, capi.JAC_ANALYTIC, 0.0)
    d = np.random.RandomState(2).uniform(-1, 1, 3 * m.nv); d[c.constraints(h, 3)] = 0.0
    vd, out = c.vec(3, d), {}
    for tma in (1, 0):
        capi.tune("tma", tma)
        s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 50, 2)
        v = c.vec(3)
        c.precond_apply(s, A, vd, v)
        out[tma] = c.download(v, 3)
    capi.tune("tma", 1)
    assert np.linalg.norm(out[1] - out[0]) <= 1e-11 * np.linalg.norm(out[0])
