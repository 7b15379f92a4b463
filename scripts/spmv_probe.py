"""Times the fine-level star SpMV kernels of a linear-problem step (CUDA events around every launch, pnp_profile_spmv) for
each kernel variant selected through pnp_tune: plain y = A x, residual b - A x, smoother step.  The matrix is the
work-space Jacobian the solver assembles, so jac_compact selects its layout: 5 value planes (the default on pore.cfg) or
7 (jac_compact=0).  The residual and smoother of the finest multigrid level read the single-precision copy of its
planes where mg_f32_min_rows selects it (default: levels of 2^22 rows and more; mg_f32_min_rows=1e30: none).  k = 7 by
default (141 M dofs).  The line "copy" is the device-to-device copy bandwidth measured in the same process (CUDA events,
2 x 4 GiB per copy), the yardstick of the GB/s figures.
  python scripts/spmv_probe.py [levels] [variant ...]     variant = name=value[,name=value...]   e.g. tma=0 tma=1,tma_stages=2
"""
import os
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import json  # noqa: E402

import util  # noqa: E402
from dune_pnp_b200 import capi  # noqa: E402

DEFAULTS = {"tma": 1, "tma_stages": 2, "tma_lpr": 2, "jac_compact": 1, "mg_f32_min_rows": -1}
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


def copy_gbs():
    import torch
    a = torch.empty(1 << 29, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        b.copy_(a)
    e0.record()
    for _ in range(20):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 20 * 2 * a.numel() * 8 / (e0.elapsed_time(e1) / 1e3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


print("copy", json.dumps({"GB/s": round(copy_gbs(), 1)}), flush=True)
s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 3, 2)  # one hierarchy for all variants (its set-up follows the knobs)
for var in variants:
    knobs = dict(DEFAULTS)
    for kv in var.split(","):
        k, v = kv.split("=")
        knobs[k] = float(v)
    for k, v in knobs.items():
        capi.tune(k, v)
    planes = 5 if knobs["jac_compact"] else 7  # (pore.cfg and the Jacobi-smoothed multigrid qualify for the compact layout)
    base = (8 * planes + 4) * ns + 52 * nv
    thr = knobs["mg_f32_min_rows"]
    f32 = knobs["tma"] and nv >= (thr if thr >= 0 else 1 << 22)
    mg = base - (4 * planes * ns if f32 else 0)  # the multigrid's launches: float planes where its rule gives them
    # smoother: b and the rows' own x (D^-1 is computed in the kernel)
    nbytes = {"plain": base, "residual": mg + 24 * nv, "smoother": mg + 48 * nv}
    c.vec_set(u, 0.05)
    c.slp(h, u, s, 1e-30, capi.JAC_ANALYTIC, 0.0)  # set-up + warm-up
    c.vec_set(u, 0.05)
    c.profile_spmv(True)
    c.slp(h, u, s, 1e-30, capi.JAC_ANALYTIC, 0.0)
    n, ms = c.profile_spmv_get()
    c.profile_spmv(False)
    out = {"planes": planes, "f32": bool(f32)}
    for name, cnt, t in zip(("plain", "residual", "smoother"), n, ms):
        if cnt:
            out[name] = {"launches": cnt, "avg_ms": round(t / cnt, 4), "GB": round(nbytes[name] / 1e9, 2),
                         "GB/s": round(nbytes[name] / (t / cnt) / 1e6, 1)}
    print(var, json.dumps(out), flush=True)
for k, v in DEFAULTS.items():
    capi.tune(k, v)
