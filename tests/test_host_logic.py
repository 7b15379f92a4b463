"""CPU tests of the PRODUCT's per-item logic (the __host__ __device__ functions the CUDA kernels wrap), run through
tests/host_harness against the oracle: star construction, pattern, constraints, element integrals, FD and exact
Jacobian rows, boundary terms, refinement.  Plus: the C ABI library loads and exports every declared symbol."""
import ctypes
import os
import re

import numpy as np
import pytest

import harness
import util
from oracle import binding as ora

OPS = [ora.OP_PB, ora.OP_POISSON, ora.OP_DIFFUSION, ora.OP_MASS, ora.OP_PNP]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def case(name, levels=0):
    a = util.load_mesh_arrays(name)
    m = ora.Mesh.from_arrays(**a).refine(levels)
    p = ora.Params.read(util.cfg_path(name))
    a = dict(x=m.x, y=m.y, tri=m.tri, ba=m.ba, bb=m.bb, bphys=m.bphys)
    return a, m, p


@pytest.mark.parametrize("renumber", [False, True])
@pytest.mark.parametrize("name", util.MESHES)
def test_star_pattern_and_constraints_bit_exact(name, renumber):
    a, m, p = case(name)
    S = harness.Star(a, p.surf, renumber)
    assert S.nslots == m.nv + 2 * (m.nv + m.nT - 1)  # nnz_1 = nv + 2 nE
    for F, comp0 in ((1, 0), (1, 2), (3, 0)):
        rp, col = S.export_csr(F, comp0)
        rp_o, col_o = ora.pattern(m, p, F, comp0)
        assert np.array_equal(rp, rp_o) and np.array_equal(col, col_o)
        assert np.array_equal(S.dirichlet(F, comp0), ora.dirichlet(m, p, F, comp0))


@pytest.mark.parametrize("name,levels", [("one_wall", 2), ("pore_small", 1)])
def test_refinement_rule_matches_oracle(name, levels):
    a, m0, p = case(name)
    for _ in range(levels):
        a = harness.refine(a)
    m = m0.refine(levels)
    for k in a:
        assert np.array_equal(a[k], getattr(m, k)), k


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name,levels", [("one_wall", 0), ("sphere", 0), ("cylinder", 0), ("pore_small", 1), ("pore", 0)])
def test_residual_rows_match_oracle(name, levels, op):
    a, m, p = case(name, levels)
    S = harness.Star(a, p.surf, True)
    rng = np.random.RandomState(1)
    F = ora.nfields(op)
    u = rng.uniform(-1, 1, F * m.nv); a0 = rng.uniform(0, 1, m.nv); a1 = rng.uniform(0, 1, m.nv)
    r_o, ab = ora.residual(m, p, op, u, a0, a1, valency=-1.0, want_abs=True)
    r = S.residual(op, p.sys, u, a0, a1, valency=-1.0)
    assert np.all(np.abs(r - r_o) <= 1e-12 * ab)
    # rounding level: the product takes each triangle as (v, neighbour, next neighbour) and sums over the ring
    assert np.all(np.abs(r - r_o) <= 64 * 2.3e-16 * ab)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", ["one_wall", "cylinder", "pore_small"])
def test_jacobian_rows_match_oracle(name, op, mode):
    a, m, p = case(name)
    S = harness.Star(a, p.surf, True)
    rng = np.random.RandomState(2)
    F = ora.nfields(op)
    u = rng.uniform(-1, 1, F * m.nv); a0 = rng.uniform(0, 1, m.nv); a1 = rng.uniform(0, 1, m.nv)
    rp, col, val_o, ab = ora.jacobian(m, p, op, u, a0, a1, valency=-1.0, mode=mode, eps=1e-11, want_abs=True)
    rp2, col2, val = S.jacobian(op, p.sys, u, a0, a1, valency=-1.0, mode=mode, eps=1e-11)
    assert np.array_equal(col, col2)
    assert np.all(np.abs(val - val_o) <= 1e-12 * ab + 1e-300)
    if mode == 0:
        # off-diagonal entries are two-term sums: the FD-faithful path reproduces the oracle bit for bit (same libm here)
        rows = np.repeat(np.arange(len(rp) - 1), np.diff(rp))
        off = (rows % m.nv) != (col % m.nv)  # entries coupling two different vertices
        assert np.array_equal(val[off], val_o[off])


def test_mesh_errors_are_detected():
    a, m, p = case("one_wall")
    bad = dict(a); bad["ba"], bad["bb"], bad["bphys"] = a["ba"][:-1], a["bb"][:-1], a["bphys"][:-1]
    with pytest.raises(RuntimeError, match="error 4"):   # boundary face without boundary segment
        harness.Star(bad, p.surf)
    bad = dict(a); bad["ba"] = a["ba"].copy(); bad["ba"][0] = a["tri"][10, 0]; bad["bb"] = a["bb"].copy(); bad["bb"][0] = a["tri"][10, 1]
    with pytest.raises(RuntimeError):
        harness.Star(bad, p.surf)
    # two triangles touching in one vertex only -> that vertex has two fans (non-manifold)
    bow = dict(x=np.array([0., 1, 0, -1, 0]), y=np.array([0., 1, 1, -1, -1]), tri=np.array([[0, 1, 2], [0, 3, 4]], dtype=np.int32),
               ba=np.zeros(0, np.int32), bb=np.zeros(0, np.int32), bphys=np.zeros(0, np.int32))
    with pytest.raises(RuntimeError, match="error 2"):
        harness.Star(bow, p.surf)
    deg = dict(a); deg["x"] = a["x"].copy(); deg["y"] = a["y"].copy()
    t = a["tri"][0]; deg["x"][t[2]] = deg["x"][t[1]]; deg["y"][t[2]] = deg["y"][t[1]]
    with pytest.raises(RuntimeError):
        harness.Star(deg, p.surf)


def test_c_abi_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "pnp_b200.h")).read()
    names = sorted(set(re.findall(r"\b(pnp_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) > 40
    from dune_pnp_b200 import capi
    lib = capi.lib()  # raises if the CUDA library has not been built -- there is no fallback
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from dune_pnp_b200 import capi
    with pytest.raises(capi.PnpError) as e:
        capi.Context(0)
    assert e.value.status == 6  # PNP_E_CUDA


# ---- sequential-order preconditioners, level-scheduled (pnp_sweep.cuh) vs the oracle's plain sequential sweeps ----
def _jac_case(name, levels, op):
    a, m, p = case(name, levels)
    S = harness.Star(a, p.surf, True)
    rng = np.random.RandomState(3)
    F = ora.nfields(op)
    u = rng.uniform(-0.5, 0.5, F * m.nv)
    if op == ora.OP_PNP:
        u[m.nv:] = rng.uniform(0.02, 0.1, 2 * m.nv)
    a0 = rng.uniform(0, 1, m.nv); a1 = rng.uniform(0, 1, m.nv)
    rp, col, val = S.jacobian(op, p.sys, u, a0, a1, valency=1.0, mode=1)
    return S, F, rp, col, val, rng.uniform(-1, 1, F * m.nv)


def test_sweep_levels_are_a_valid_schedule():
    S, F, rp, col, val, d = _jac_case("cylinder", 0, ora.OP_PNP)
    for full in (0, 1):
        nlev, lev = S.sweep_levels(3, full)
        lev_lex = np.zeros(3 * S.nv, dtype=np.int64)
        lev_lex.reshape(3, S.nv)[:, S.int2ext] = lev.reshape(S.nv, 3).T
        for i in range(3 * S.nv):
            cols = col[rp[i]:rp[i + 1]]
            vals_i = val[rp[i]:rp[i + 1]]
            lower = cols[(cols < i) & ((vals_i != 0) | bool(full))]
            # coupled predecessors sit on strictly lower levels, and the level is the smallest such number
            assert np.all(lev_lex[lower] < lev_lex[i])
        assert lev.min() == 0 and len(np.unique(lev)) == nlev


@pytest.mark.parametrize("steps", [1, 3])
@pytest.mark.parametrize("name,levels,op", [("one_wall", 1, ora.OP_PB), ("sphere", 0, ora.OP_POISSON), ("cylinder", 0, ora.OP_PNP),
                                            ("pore_small", 1, ora.OP_PNP), ("pore", 0, ora.OP_DIFFUSION)])
def test_level_scheduled_ssor_equals_sequential_ssor(name, levels, op, steps):
    S, F, rp, col, val, d = _jac_case(name, levels, op)
    x = S.ssor_apply(F, S.last_vals, steps, d)
    x_o = ora.prec_apply(rp, col, val, d, ora.PREC_SSOR, steps)
    assert np.linalg.norm(x - x_o) <= 1e-13 * np.linalg.norm(x_o)


@pytest.mark.parametrize("name,levels,op", [("one_wall", 1, ora.OP_PB), ("sphere", 0, ora.OP_POISSON), ("cylinder", 0, ora.OP_PNP),
                                            ("pore_small", 1, ora.OP_PNP), ("pore", 0, ora.OP_DIFFUSION)])
def test_level_scheduled_ilu0_equals_sequential_ilu0(name, levels, op):
    S, F, rp, col, val, d = _jac_case(name, levels, op)
    x = S.ilu0_apply(F, S.last_vals, d)
    x_o = ora.prec_apply(rp, col, val, d, ora.PREC_ILU0)
    assert np.linalg.norm(x - x_o) <= 1e-12 * np.linalg.norm(x_o)


@pytest.mark.parametrize("example", ["stationary_pnp", "stationary_pnp_from_pb", "instationary_pnp_md"])
def test_facade_examples_compile(example):
    """The PDELab-named C++ facade and the two driver rewrites compile against the C ABI header (no CUDA needed)."""
    import subprocess
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", example + ".cc")])


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line with the contract's keys,
    same metric / unit as the GPU arm, zero transfer bytes."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-level", "2", "--cpu-threads", "2"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "newton_step_dofs_per_s" and line["unit"] == "DOF/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in line
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 2 and line["value"] > 0
    # per-phase timers of the multi-core run and the single-core run beside it (BASELINE.md section 4)
    for ph in ("jacobian_fd", "residual", "krylov_iteration", "spmv"):
        assert cb["phases_s"][ph] > 0 and cb["single_core"]["phases_s"][ph] > 0
    assert line["config"]["levels"] == 2 and line["config"]["dofs"] == 139959
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["dtype"] == "f64"
    # ranks other than 0 stay silent under torchrun
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_dump_outputs_writes_a_fixed_sample_within_64_mb(tmp_path):
    """`bench.py --dump-outputs`: a small state is written whole; a larger one as the same seeded, sorted vertex sample on
    every call (all three fields of each sampled vertex), float64, at most 64 MB in all."""
    import bench
    from dune_pnp_b200 import capi
    r = capi.NewtonResult()
    r.converged, r.iterations, r.first_defect, r.defect, r.linear_iterations = 0, 1, 3.4, 1.5e-5, 5
    small = np.arange(3 * 1000, dtype=np.float64)
    bench.dump_outputs(str(tmp_path / "s"), small, r)
    assert np.array_equal(np.load(tmp_path / "s" / "u.npy"), small.reshape(3, -1))
    res = np.load(tmp_path / "s" / "newton_result.npy")
    assert res.dtype == np.float64 and list(res[:4]) == [0, 1, 3.4, 1.5e-5] and res[5] == 5
    nv = bench.DUMP_VERTICES + 12345
    big = np.arange(3 * nv, dtype=np.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big, r)
    a, b = np.load(tmp_path / "a" / "u.npy"), np.load(tmp_path / "b" / "u.npy")
    assert a.dtype == np.float64 and a.shape == (3, bench.DUMP_VERTICES) and np.array_equal(a, b)
    idx = a[0].astype(np.int64)
    assert np.all(np.diff(idx) > 0) and np.array_equal(a[1], idx + nv) and np.array_equal(a[2], idx + 2 * nv)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64e6


def test_shared_sinh_is_bit_identical_on_both_sides_and_accurate():
    """SURVEY H1: the PB source term's sinh is one sequence of +, -, *, /, floor on the device (pnp_elem.cuh: pnp_sinh,
    compiled here for the host without FMA contraction) and in the oracle (sinh_shared): same bits, within 4 ulp of libm."""
    import ctypes as C
    rng = np.random.RandomState(0)
    x = np.concatenate([rng.uniform(-0.5, 0.5, 20000), rng.uniform(-30, 30, 20000), rng.uniform(-600, 600, 2000),
                        [0.0, -0.0, 0.35, -0.35, 0.34999999999999, 1e-300, 1e-9, 709.0 * 0.98]])
    y_dev = np.zeros_like(x)
    harness.lib().hh_sinh(len(x), x.ctypes.data_as(C.POINTER(C.c_double)), y_dev.ctypes.data_as(C.POINTER(C.c_double)))
    y_ora = ora.sinh_shared(x)
    assert np.array_equal(y_dev.view(np.int64), y_ora.view(np.int64))
    ref = np.sinh(x)
    ulp = np.abs(y_ora - ref) / np.maximum(np.spacing(np.abs(ref)), 5e-324)
    assert ulp.max() <= 4.0
    assert np.array_equal(np.signbit(y_ora), np.signbit(x))
