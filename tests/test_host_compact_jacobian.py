"""CPU tests of the compact 5-plane PNP Jacobian layout (dune_pnp_b200/csrc/pnp_elem.cuh, pnp_star.cuh): on random triangles of
both orientations and random states, the compact rows and their expansion into 3x3 block entries reproduce the 7-plane exact
derivative -- the planes they share bit for bit, the two diagonal blocks rebuilt from L and D to a few ulp of |L| + |D| --
and the layout rule keeps 7 planes wherever a surface constrains some components and not others."""
import configparser
import ctypes as C
import glob
import itertools
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_harness", "compact_jacobian.cpp")
JAC_FD_FAITHFUL, JAC_ANALYTIC = 0, 1
BTYPE_KEYS = ("coulombBtype", "plusDiffusionBtype", "minusDiffusionBtype")

_dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("compact") / "libcompact.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++", SRC, "-o", so])
    L = C.CDLL(so)
    L.hc_jacobian_planes.restype = C.c_int
    return L


def rows(lib, xy, xl, phys, I):
    full, compact, expanded = np.zeros(21), np.zeros(15), np.zeros(21)
    args = [np.ascontiguousarray(a, dtype=np.float64) for a in (xy, xl, phys)]
    lib.hc_rows(*[a.ctypes.data_as(_dp) for a in args], C.c_int(I), full.ctypes.data_as(_dp), compact.ctypes.data_as(_dp),
                expanded.ctypes.data_as(_dp))
    return full.reshape(3, 7), compact.reshape(3, 5), expanded.reshape(3, 7)


@pytest.mark.parametrize("cylindrical", [0, 1])
def test_compact_rows_reproduce_seven_planes(lib, cylindrical):
    rng = np.random.RandomState(7 + cylindrical)
    phys = np.array([3.1415, 0.7, 0.06, 1.0, cylindrical])
    for trial in range(40):
        base = np.array([[0.1, 0.2], [1.3, 0.5], [0.4, 1.7]]) + 0.3 * rng.uniform(-1, 1, (3, 2))
        # states of the size a Newton iterate has: potential up to tens, concentrations around c0
        xl = np.concatenate([rng.uniform(-30, 30, 3), rng.uniform(0, 0.2, 6)])
        for perm in itertools.permutations(range(3)):  # both orientations, every element-local vertex order
            xy = base[list(perm)].ravel()
            for I in range(3):
                full, compact, expanded = rows(lib, xy, xl, phys, I)
                # L, M, (c+,phi), (c-,phi): the same operations as the 7-plane planes 0, 1, 3, 5
                assert np.array_equal(compact[:, :4], full[:, [0, 1, 3, 5]])
                # (phi,c-) is the exact negation of M
                assert np.array_equal(compact[:, 1], -full[:, 2])
                assert np.array_equal(expanded[:, [0, 1, 2, 3, 5]], full[:, [0, 1, 2, 3, 5]])
                # (c+,c+) = L - D and (c-,c-) = L + D up to the rounding of reordered sums
                scale = np.abs(compact[:, 0]) + np.abs(compact[:, 4])
                ulp = np.spacing(scale)
                for p in (4, 6):
                    err = np.abs(expanded[:, p] - full[:, p])
                    assert np.all(err <= 8 * ulp), (trial, perm, I, p, err / ulp)


def surface_btypes(text):
    cp = configparser.ConfigParser(strict=False)
    cp.optionxform = str
    cp.read_string(text)
    n = int(cp["system"]["n_surfaces"])
    return [int(cp["surface_%d" % s][k]) for s in range(n) for k in BTYPE_KEYS]


def planes(lib, btype, mode=JAC_ANALYTIC, degree=1, solver_ok=True):
    arr = (C.c_int * max(len(btype), 1))(*btype)
    return lib.hc_jacobian_planes(mode, degree, int(solver_ok), arr, len(btype) // 3)


MIXED_CFG = """
[system]
n_surfaces=2
[surface_0]
coulombBtype=1
plusDiffusionBtype=1
minusDiffusionBtype=1
[surface_1]
coulombBtype=0
coulombPotential=0
plusDiffusionBtype=1
plusDiffusionFlux=0
minusDiffusionBtype=1
minusDiffusionFlux=0
"""


def test_layout_rule(lib):
    cfgs = sorted(glob.glob(os.path.join(HERE, "golden", "*.cfg")))
    assert cfgs
    for path in cfgs:  # every shipped configuration constrains its surfaces' components together
        with open(path) as f:
            bt = surface_btypes(f.read())
        assert planes(lib, bt) == 5, path
        assert planes(lib, bt, mode=JAC_FD_FAITHFUL) == 7
        assert planes(lib, bt, degree=2) == 7
        assert planes(lib, bt, solver_ok=False) == 7
    # a Dirichlet potential beside Neumann concentrations: (c+,c+) and (phi,phi) are masked differently
    assert planes(lib, surface_btypes(MIXED_CFG)) == 7
