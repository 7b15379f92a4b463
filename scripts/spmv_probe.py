"""Times the fine-level star SpMV kernels of a linear-problem step (CUDA events around every launch, pnp_profile_spmv) for
each kernel variant selected through pnp_tune: plain y = A x, residual b - A x, smoother step.  The matrix is the
work-space Jacobian the solver assembles, so jac_compact selects its layout: 5 value planes (the default on pore.cfg) or
7 (jac_compact=0).  k = 7 by default (141 M dofs).
  python scripts/spmv_probe.py [levels] [variant ...]     variant = name=value[,name=value...]   e.g. tma=0 tma=1,tma_stages=2
"""
import os
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import json  # noqa: E402

import util  # noqa: E402
from dune_pnp_b200 import capi  # noqa: E402

DEFAULTS = {"tma": 1, "tma_stages": 2, "jac_compact": 1}
levels = int(sys.argv[1]) if len(sys.argv) > 1 else 7
variants = sys.argv[2:] or ["tma=1,tma_stages=3", "tma=1,tma_stages=2", "jac_compact=0,tma_stages=2"]
c = capi.Context(0)
c.mesh_set(**util.load_mesh_arrays("pore")); c.params_read(util.cfg_path("pore"))
c.mesh_refine(levels); c.mesh_finalize(True)
sz = c.mesh_sizes()
nv, ns = sz["nv"], sz["nslots"]
h = c.operator(capi.OP_PNP, 0)
u = c.vec(3)
print("levels %d nv %d nslots %d" % (levels, nv, ns), flush=True)
for var in variants:
    knobs = dict(DEFAULTS)
    for kv in var.split(","):
        k, v = kv.split("=")
        knobs[k] = float(v)
    for k, v in knobs.items():
        capi.tune(k, v)
    planes = 5 if knobs["jac_compact"] else 7  # (pore.cfg and the Jacobi-smoothed multigrid qualify for the compact layout)
    base = (8 * planes + 4) * ns + 52 * nv
    # smoother: b and the rows' own x (D^-1 is computed in the kernel)
    nbytes = {"plain": base, "residual": base + 24 * nv, "smoother": base + 48 * nv}
    s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 3, 2)
    c.vec_set(u, 0.05)
    c.slp(h, u, s, 1e-30, capi.JAC_ANALYTIC, 0.0)  # set-up + warm-up
    c.vec_set(u, 0.05)
    c.profile_spmv(True)
    c.slp(h, u, s, 1e-30, capi.JAC_ANALYTIC, 0.0)
    n, ms = c.profile_spmv_get()
    c.profile_spmv(False)
    out = {"planes": planes}
    for name, cnt, t in zip(("plain", "residual", "smoother"), n, ms):
        if cnt:
            out[name] = {"launches": cnt, "avg_ms": round(t / cnt, 4), "GB/s": round(nbytes[name] / (t / cnt) / 1e6, 1)}
    print(var, json.dumps(out), flush=True)
for k, v in DEFAULTS.items():
    capi.tune(k, v)
