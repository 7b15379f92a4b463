"""GPU tests of the compact 5-plane PNP Jacobian that Newton and the linear-problem solver assemble where it applies
(pnp_tune "jac_compact" = 1, the default) against the 7-plane layout (jac_compact = 0), in one process:

  * on the refined pore mesh, levels 4 and 5, with a smooth state: one BiCGSTAB iteration without preconditioner, with
    Jacobi and with the multigrid (plain, residual and smoother-step SpMVs, Galerkin and re-discretised levels, dense
    coarsest solve) gives the same correction up to rounding, and a multigrid-preconditioned solve takes as many
    iterations with either layout;
  * where the compact layout does not apply -- a surface with a Dirichlet potential and Neumann concentrations, the
    FD-faithful Jacobian, an SSOR preconditioner -- the knob changes nothing: results are bit-identical.
"""
import os

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu


def _capi():
    from dune_pnp_b200 import capi
    return capi


@pytest.fixture
def compact_knob():
    capi = _capi()
    yield lambda on: capi.tune("jac_compact", 1 if on else 0)
    capi.tune("jac_compact", 1)


def pore_ctx(levels, cfg=None):
    capi = _capi()
    c = capi.Context(0)
    c.mesh_set(**util.load_mesh_arrays("pore"))
    c.params_read(cfg or util.cfg_path("pore"))
    c.mesh_refine(levels)
    c.mesh_finalize(True)
    return c


def smooth_state(c):
    m = c.mesh_get()
    x, y = m["x"], m["y"]
    sx, sy = np.ptp(x), np.ptp(y)
    phi = 5.0 * np.sin(2.0 * x / sx) * np.cos(y / sy)
    cp = 0.06 * (1.0 + 0.3 * np.cos(3.0 * y / sy))
    cm = 0.06 * (1.0 - 0.2 * np.sin(2.0 * x / sx + y / sy))
    return np.concatenate([phi, cp, cm])


def slp_step(c, u0, prec, maxit, reduction, prec_steps=2):
    capi = _capi()
    h = c.operator(capi.OP_PNP, 0)
    u = c.vec(3, u0)
    s = c.solver(capi.SOLVER_BCGS, prec, maxit, prec_steps)
    res = c.slp(h, u, s, reduction, jac_mode=capi.JAC_ANALYTIC, eps=0.0)
    return u0 - c.download(u, 3), res


@pytest.mark.parametrize("levels", [4, 5])
def test_compact_layout_same_correction(levels, compact_knob):
    capi = _capi()
    c = pore_ctx(levels)
    u0 = smooth_state(c)
    for prec, tol in ((capi.PREC_NONE, 1e-12), (capi.PREC_JACOBI, 1e-12), (capi.PREC_AMG, 1e-10)):
        z = {}
        for on in (0, 1):
            compact_knob(on)
            z[on], _ = slp_step(c, u0, prec, 1, 1e-30)
        assert np.all(np.isfinite(z[1])) and np.linalg.norm(z[0]) > 0
        for k in range(3):  # per field
            a, b = z[0].reshape(3, -1)[k], z[1].reshape(3, -1)[k]
            rel = np.linalg.norm(b - a) / max(np.linalg.norm(a), 1e-300)
            assert rel <= tol, (prec, k, rel)


@pytest.mark.parametrize("levels", [4, 5])
def test_compact_layout_same_iterations(levels, compact_knob):
    capi = _capi()
    c = pore_ctx(levels)
    u0 = smooth_state(c)
    its = {}
    for on in (0, 1):
        compact_knob(on)
        _, res = slp_step(c, u0, capi.PREC_AMG, 20000, 1e-8)
        assert res.converged
        its[on] = res.iterations
    assert its[0] == its[1]


def mixed_cfg(tmp_path):
    """pore.cfg with Neumann concentrations on the surface whose potential is Dirichlet (surface_3)."""
    with open(util.cfg_path("pore")) as f:
        text = f.read()
    old = ("plusDiffusionBtype=0\nplusDiffusionConcentration=0.06\nminusDiffusionBtype=0\nminusDiffusionConcentration=0.06\n\n"
           "[surface_4]")
    assert old in text
    text = text.replace(old, "plusDiffusionBtype=1\nplusDiffusionFlux=0\nminusDiffusionBtype=1\nminusDiffusionFlux=0\n\n[surface_4]")
    path = os.path.join(str(tmp_path), "pore_mixed.cfg")
    with open(path, "w") as f:
        f.write(text)
    return path


@pytest.mark.parametrize("case", ["mixed_masks", "fd_faithful", "ssor"])
def test_layout_not_applicable_is_bit_identical(case, compact_knob, tmp_path):
    capi = _capi()
    c = pore_ctx(2, mixed_cfg(tmp_path) if case == "mixed_masks" else None)
    u0 = smooth_state(c)
    jac = capi.JAC_FD_FAITHFUL if case == "fd_faithful" else capi.JAC_ANALYTIC
    prec = capi.PREC_SSOR if case == "ssor" else capi.PREC_AMG
    out = {}
    for on in (0, 1):
        compact_knob(on)
        h = c.operator(capi.OP_PNP, 0)
        u = c.vec(3, u0)
        st, res = c.newton(h, u, c.solver(capi.SOLVER_BCGS, prec, 2000, 1), c.newton_opts(jac_mode=jac, max_iterations=2),
                           check=False)
        out[on] = (c.download(u, 3), res.iterations, res.linear_iterations, res.defect)
    assert np.array_equal(out[0][0], out[1][0])
    assert out[0][1:] == out[1][1:]
