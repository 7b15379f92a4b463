#!/usr/bin/env python
"""bench.py -- one PNP Newton step (Jacobian assembly + preconditioned BiCGSTAB solve + line search) on the
uniformly refined pore mesh (BASELINE.json configs[4]: test/pore_pnp refined to >= 50 M dofs).

A "step" is one Newton iteration of the monolithic 3-field PNP system (stationary_pnp.hh:280-294) started from
the same state u_s every time: u_s is the PNP solution converged on refinement level `--coarse-level` (reference
flow: PB Newton -> interpolate(BCExtension) -> PNP Newton) and carried to the fine mesh by P1 interpolation
(nested iteration), i.e. a late Newton step of a production run.  value = dofs / step time.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--levels L] [--impl reference] [--dump-outputs DIR]

N > 1 (torchrun, one rank per GPU): the SAME global problem is split into N subdomains (strong scaling); NCCL carries
halo values and scalar sums only (DESIGN.md "multi-GPU").
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "newton_step_dofs_per_s"
UNIT = "DOF/s"


def load_case():
    import util
    return util.load_mesh_arrays("pore"), util.cfg_path("pore")


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill(); out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (a port of the reference's algorithm; the reference itself needs DUNE and cannot be built)
# ------------------------------------------------------------------------------------------------------------
def carry_numpy(m_coarse, u_lex, F):
    """P1 interpolation of nodal fields to the once-refined mesh (oracle's refinement rule)."""
    tri = m_coarse.tri.astype(np.int64)
    e = np.concatenate([tri[:, [0, 1]], tri[:, [0, 2]], tri[:, [1, 2]]])
    lo, hi = e.min(1), e.max(1)
    keys = np.unique((lo << 32) | hi)
    a, b = (keys >> 32).astype(np.int64), (keys & 0xffffffff).astype(np.int64)
    u = u_lex.reshape(F, m_coarse.nv)
    return np.concatenate([u, 0.5 * (u[:, a] + u[:, b])], axis=1).reshape(-1)


_CPU_STATE = {}


def cpu_setup(level):
    """Oracle objects for the CPU arm at refinement level `level` of the pore mesh (cached): mesh, pattern, incidence lists
    and the start state -- the state after the first PNP Newton iteration on the unrefined mesh
    (tests/golden/pore_solution.npz, scripts/make_golden_solutions.py), P1-interpolated `level` times."""
    if level in _CPU_STATE:
        return _CPU_STATE[level]
    from oracle import binding as ora
    import util
    a, cfg = load_case()
    p = ora.Params.read(cfg)
    m = ora.Mesh.from_arrays(**a)
    u = np.load(os.path.join(util.GOLDEN, "pore_solution.npz"))["u1"]
    for _ in range(level):
        u = carry_numpy(m, u, 3)
        m = m.refine(1)
    _CPU_STATE[level] = (ora.Bench(m, p, ora.OP_PNP), m, u)
    return _CPU_STATE[level]


def cpu_newton_step(level=5, threads=1, krylov_iters=5):
    """One BOUNDED sample of the reference's Newton step on the host (the oracle; DUNE itself cannot be built here): the
    reference's own jacobian_volume (NumericalJacobianVolume, eps 1e-11), two residual assemblies (defect + one line-search
    trial) and `krylov_iters` iterations of its default backend BiCGSTAB + SSOR(1) (instationary_pnp_from_pb_md.hh:188-191).
    The Krylov budget is what the GPU step needs with its multigrid (5); BiCGSTAB + SSOR(1) needs 1 440 iterations for
    this step on the unrefined mesh and more on every finer one, so the sample is a LOWER bound of the reference's step
    time.  threads > 1: element / row loops and vector operations on that many cores (OpenMP), SSOR sweeps sequential."""
    b, m, u = cpu_setup(level)
    r = b.step(u, threads=threads, jac_mode=0, krylov_iters=krylov_iters)
    dofs = 3 * m.nv
    nnz = b.nnz
    return dict(dofs=dofs, level=level, threads=threads, seconds=r["total_s"], value=dofs / r["total_s"],
                phases_s={"jacobian_fd": r["jacobian_s"], "residual": r["residual_s"], "krylov_iteration": r["krylov_s"] / max(r["krylov_iterations"], 1),
                          "spmv": r["spmv_s"]},
                spmv_gbs=(12.0 * nnz + 20.0 * dofs) / r["spmv_s"] / 1e9, assembled_dofs_per_s=dofs / (r["jacobian_s"] + r["residual_s"]),
                krylov_iterations=r["krylov_iterations"])


def cpu_sample_text(r):
    return ("oracle (CPU restatement of the reference path), pore mesh refined %d times (%d dofs), %d thread(s): FD Jacobian %.2f s + "
            "2 residuals x %.2f s + %d BiCGSTAB/SSOR(1) iterations x %.2f s (budget = the GPU step's iteration count; the "
            "reference's solver needs >= 1 440: lower bound of its step time); SpMV %.1f GB/s" % (
                r["level"], r["dofs"], r["threads"], r["phases_s"]["jacobian_fd"], r["phases_s"]["residual"], r["krylov_iterations"],
                r["phases_s"]["krylov_iteration"], r["spmv_gbs"]))


def run_reference(args, rank):
    if rank != 0:
        return
    from oracle import binding as ora
    threads = args.cpu_threads if args.cpu_threads > 0 else ora.max_threads()
    # the sample is sized so that W + K steps end within a few minutes: ~20 s per step at level 5 on 8 cores, ~5 s at level 4
    # (DOF/s barely depends on the level: every phase is linear in the mesh size)
    level = args.cpu_level if args.cpu_level >= 0 else (5 if args.warmup + args.steps <= 8 else 4)
    cpu_setup(level)
    res = [cpu_newton_step(level, threads) for _ in range(args.warmup + args.steps)][args.warmup:]
    t = float(np.mean([r["seconds"] for r in res]))
    r = res[-1]
    one = cpu_newton_step(level, 1)   # the single-core figures beside it
    line = {"impl": "reference", "metric": METRIC, "value": r["dofs"] / t, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "test/pore_pnp (pore.msh + pore.cfg) uniformly refined %d times: bounded sample of one monolithic PNP "
                                   "Newton step on the host cores" % r["level"], "levels": r["level"], "dofs": r["dofs"]},
            "cpu_baseline": {"value": r["dofs"] / t, "unit": UNIT, "cores": threads, "kind": "port", "sample": cpu_sample_text(r),
                             "phases_s": r["phases_s"], "assembled_dofs_per_s": r["assembled_dofs_per_s"], "spmv_gbs": r["spmv_gbs"],
                             "single_core": {"value": one["value"], "phases_s": one["phases_s"], "assembled_dofs_per_s": one["assembled_dofs_per_s"],
                                             "spmv_gbs": one["spmv_gbs"]}},
            "e2e": {"value": r["dofs"] / t, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def coarse_stage(c, capi, coarse_level, jac_mode, prec_steps, verbose):
    """Reference flow on the coarse level: PB Newton -> interpolate(BCExtension) -> PNP Newton. Returns the 3-field vector."""
    def solver():
        # plain aggregation AMG V(2,2): it survives the convection-dominated first Newton step of the reference flow
        # (discontinuous initial guess at the outflow Dirichlet boundary)
        s_ = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 20000, prec_steps, 0)
        c.solver_set_option(s_, "amg_geometric", 0)
        return s_
    c.mesh_refine(coarse_level); c.mesh_finalize(True)
    hpb = c.operator(capi.OP_PB, 0)
    vpb = c.vec(1)
    c.newton(hpb, vpb, solver(), c.newton_opts(jac_mode=jac_mode))
    f = [c.vec(1) for _ in range(3)]
    for k in range(3):
        c.interpolate_bcext(k, vpb, f[k])
    vu = c.vec(3); c.pack3(vu, *f)
    h = c.operator(capi.OP_PNP, 0)
    st, r = c.newton(h, vu, solver(), c.newton_opts(jac_mode=jac_mode))
    if verbose:
        print("# coarse level %d: PNP Newton %d its, linear %s" % (coarse_level, r.iterations,
              list(r.linear_iterations_history[:r.n_history])), file=sys.stderr, flush=True)
    return vu


def build_state(c, capi, levels, coarse_level, jac_mode, prec_steps, verbose):
    """N = 1: coarse solve, then nested iteration to the fine mesh on the device. Returns (op, solver, u_s)."""
    vu = coarse_stage(c, capi, coarse_level, jac_mode, prec_steps, verbose)
    c.carry_set([vu])
    c.mesh_refine(levels - coarse_level); c.mesh_finalize(True)
    us = c.vec(3); c.carry_get(0, us)
    return c.operator(capi.OP_PNP, 0), fine_solver(c, capi, prec_steps), us


# N > 1: per-subdomain aggregation AMG V-cycle (no geometric levels across ranks yet; a truncated W-cycle halves the
# iteration count but is launch-bound on the small levels: 166 its / 15.4 s vs 300 its / 4.0 s at k = 6, N = 2)
AMG_PARTITIONED = {"amg_geometric": 0}
EXTRA_SOLVER_OPTS = {}            # --solver-opt NAME=VALUE
DENSE_COARSE = False              # --dense-coarse
PYTHON_PARTITIONER = False        # --python-partitioner
REPLICA_LEVEL = 3                 # --replica-level: N > 1, refinement level at which the hierarchy stops being distributed
AMG_FINE = {"amg_geometric": 1}   # refinement levels as multigrid levels (P1 interpolation), aggregation below the coarsest mesh


def fine_solver(c, capi, prec_steps, options=None):
    """BiCGSTAB + multigrid for the timed step: V(nu,nu) damped Jacobi; the mesh levels created by pnp_mesh_refine are the
    upper multigrid levels (P1 interpolation, Galerkin operators), aggregation AMG continues below the Gmsh mesh."""
    s = c.solver(capi.SOLVER_BCGS, capi.PREC_AMG, 20000, prec_steps, 0)
    for k, v in list((AMG_FINE if options is None else options).items()) + list(EXTRA_SOLVER_OPTS.items()):
        c.solver_set_option(s, k, v)
    return s


def build_state_partitioned(c, capi, levels, coarse_level, jac_mode, prec_steps, verbose, rank, world, dist, cfg):
    """N > 1: every rank solves the (small) coarse problem; the Gmsh mesh is partitioned, every rank refines its part level
    by level (host plumbing, dune_pnp_b200/partition.py) and registers each level as a multigrid level of the library
    (distributed geometric multigrid: halo exchange per level, re-discretised coarse operators, replicated dense solve
    on the Gmsh mesh).  The start state is the coarse solution, injected at `coarse_level` and P1-interpolated upwards."""
    from dune_pnp_b200 import partition
    a_base = c.mesh_get()                        # level 0 (the context still holds the Gmsh mesh)
    vu = coarse_stage(c, capi, coarse_level, jac_mode, prec_steps, verbose)
    ak = c.mesh_get()
    uk = c.download(vu, 3).reshape(3, -1)
    lookup_tab = {k: i for i, k in enumerate(partition._coord_keys(ak["x"], ak["y"]))}

    def lookup(x, y):
        idx = np.array([lookup_tab[k] for k in partition._coord_keys(x, y)], dtype=np.int64)
        return {"u": uk[:, idx]}

    def all_gather(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out
    # the library's native partitioner (csrc/pnp_partition.cu); --python-partitioner: its numpy cross-check (same plans)
    build = partition.build_hierarchy if PYTHON_PARTITIONER else partition.build_hierarchy_native
    plans = build(a_base, world, rank, levels, all_gather=all_gather, fields_at=(coarse_level, lookup))
    uid = [capi.Context.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    # the hierarchy is distributed down to refinement level REPLICA_LEVEL; that level is gathered to a replica of the whole
    # level mesh on every rank, below which the one-GPU hierarchy continues (refinement levels, aggregation levels, small
    # dense LU): the cycle equals the N = 1 cycle and the small levels need no halo exchanges.
    # (--dense-coarse: replicated dense LU of the 9 144-dof Gmsh system instead, ~57 ms per Newton step on every rank)
    children = partition.setup_distributed(capi, c, plans, cfg, rank, world, uid[0], replica_mesh=None if DENSE_COARSE else a_base,
                                           replica_level=0 if DENSE_COARSE else max(0, min(REPLICA_LEVEL, levels - 1)))
    fine = plans[-1]
    us = c.vec(3, fine.fields["u"].reshape(-1))
    if verbose:
        print("# rank %d: %d owned + %d ghost vertices, %d neighbours, %d multigrid levels" % (
            rank, fine.n_own, fine.nv - fine.n_own, len(fine.nbr), len(plans)), file=sys.stderr, flush=True)
    return c.operator(capi.OP_PNP, 0), fine_solver(c, capi, prec_steps), us, (children, fine)


def parity_vs_n1(args, c, capi, u_vec, fine, rank, world, dist, torch, cfg, a, jac_mode):
    """Relative L2 distance between the N-rank step result and the 1-rank result of the same step (rank 0 runs the whole
    problem once more on its own GPU, outside every timed region).  Vertices are matched by their bitwise coordinates:
    both sides are sorted lexicographically by (x, y) bit patterns on the device."""
    def sort_xy(xb, yb):
        i1 = torch.argsort(yb, stable=True)
        i2 = torch.argsort(xb[i1], stable=True)
        return i1[i2]
    n_own = fine.n_own
    dev = torch.device("cuda")
    xb = torch.from_numpy(np.ascontiguousarray(fine.x[:n_own]).view(np.int64)).to(dev)
    yb = torch.from_numpy(np.ascontiguousarray(fine.y[:n_own]).view(np.int64)).to(dev)
    uo = torch.from_numpy(c.download(u_vec, 3).reshape(3, -1)[:, :n_own].copy()).to(dev)
    counts = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(counts, torch.tensor([n_own], dtype=torch.int64, device=dev))
    counts = [int(t.item()) for t in counts]
    if rank != 0:
        dist.send(xb, 0); dist.send(yb, 0); dist.send(uo.contiguous(), 0)
        out = torch.zeros(1, dtype=torch.float64, device=dev)
        dist.broadcast(out, 0)
        return float(out.item())
    X, Y, U = [xb], [yb], [uo]
    for r in range(1, world):
        tx = torch.empty(counts[r], dtype=torch.int64, device=dev); ty = torch.empty_like(tx)
        tu = torch.empty((3, counts[r]), dtype=torch.float64, device=dev)
        dist.recv(tx, r); dist.recv(ty, r); dist.recv(tu, r)
        X.append(tx); Y.append(ty); U.append(tu)
    X, Y, U = torch.cat(X), torch.cat(Y), torch.cat(U, dim=1)
    o = sort_xy(X, Y)
    Xs, Ys, U = X[o], Y[o], U[:, o]
    del X, Y, o
    # the 1-rank run of the same step
    c1 = capi.Context(torch.cuda.current_device())
    c1.mesh_set(**a); c1.params_read(cfg)
    h1, s1, us1 = build_state(c1, capi, args.levels, args.coarse_level, jac_mode, args.prec_steps, False)
    u1 = c1.vec(3); c1.vec_copy(u1, us1)
    st, r1 = c1.newton(h1, u1, s1, c1.newton_opts(jac_mode=jac_mode, max_iterations=1), check=False)
    g = c1.mesh_get()
    ref = torch.from_numpy(c1.download(u1, 3).reshape(3, -1)).to(dev)
    c1.close()
    x1 = torch.from_numpy(g["x"].view(np.int64)).to(dev); y1 = torch.from_numpy(g["y"].view(np.int64)).to(dev)
    o1 = sort_xy(x1, y1)
    assert len(o1) == U.shape[1] and bool(torch.equal(x1[o1], Xs)) and bool(torch.equal(y1[o1], Ys)), "owned vertices of all ranks must tile the global mesh"
    ref = ref[:, o1]
    val = float((torch.linalg.norm(U - ref) / torch.linalg.norm(ref)).item())
    dist.broadcast(torch.tensor([val], dtype=torch.float64, device=dev), 0)
    return val


DUMP_VERTICES = 1 << 21   # --dump-outputs: at most this many vertices of u (3 x 8 B each, 48 MiB)


def dump_outputs(path, u, r):
    """--dump-outputs: what a caller of the timed step receives from its last call, so that two builds can be compared output
    for output.  u.npy: the updated state as (3, nv) float64 (phi, c+, c- in mesh vertex order); on meshes with more than
    DUMP_VERTICES vertices, the columns of a fixed seeded sample of vertices (sorted, the same on every run).
    newton_result.npy: converged, iterations, first defect, defect, reduction, linear iterations, line-search trials,
    Jacobian assemblies, residual assemblies (float64)."""
    os.makedirs(path, exist_ok=True)
    u = np.asarray(u, dtype=np.float64).reshape(3, -1)
    if u.shape[1] > DUMP_VERTICES:
        u = u[:, np.sort(np.random.default_rng(0).choice(u.shape[1], DUMP_VERTICES, replace=False))]
    np.save(os.path.join(path, "u.npy"), np.ascontiguousarray(u))
    np.save(os.path.join(path, "newton_result.npy"), np.array(
        [r.converged, r.iterations, r.first_defect, r.defect, r.reduction, r.linear_iterations, r.line_search_trials,
         r.jacobian_assemblies, r.residual_assemblies], dtype=np.float64))


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from dune_pnp_b200 import capi
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    a, cfg = load_case()
    c = capi.Context(local_rank)
    c.mesh_set(**a); c.params_read(cfg)
    jac_mode = capi.JAC_FD_FAITHFUL if args.jac == "fd" else capi.JAC_ANALYTIC
    t_setup = time.perf_counter()
    if world == 1:
        h, s, us = build_state(c, capi, args.levels, args.coarse_level, jac_mode, args.prec_steps, args.verbose)
    else:
        h, s, us, (_children, fine_plan) = build_state_partitioned(c, capi, args.levels, args.coarse_level, jac_mode, args.prec_steps,
                                                                   args.verbose, rank, world, dist, cfg)
    sizes = c.mesh_sizes()
    nv, ns = sizes["nv"], sizes["nslots"]       # local vertices (owned + ghost), local matrix slots
    n_own = c.mesh_owned()
    ndof = 3 * nv                                # local vector length (host buffers of the end-to-end leg)
    tot = torch.tensor([3 * n_own, ns, sizes["nT"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tot)
    gdof, gslots = int(tot[0].item()), int(tot[1].item())
    t_setup = time.perf_counter() - t_setup
    u = c.vec(3)
    opts = c.newton_opts(jac_mode=jac_mode, max_iterations=1)
    # pinned host buffers for the end-to-end leg
    h_in = torch.empty(ndof, dtype=torch.float64, pin_memory=True).numpy()
    h_out = torch.empty(ndof, dtype=torch.float64, pin_memory=True).numpy()
    h_in[:] = c.download(us, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(e2e):
        if e2e:
            c.upload(u, h_in)
        else:
            c.vec_copy(u, us)
        st, r = c.newton(h, u, s, opts, check=False)
        if st not in (0, 1):
            raise RuntimeError("Newton step failed with status %d" % st)
        if e2e:
            lib = capi.lib()
            c._ck(lib.pnp_vec_download(c._h, u, h_out.ctypes.data_as(capi._dp)))
        return r

    for _ in range(args.warmup):
        r = step(False)
    # ---- timed region: K steps, inputs resident in HBM ----
    sampler = ClockSampler(local_rank) if rank == 0 else None
    c.profile_spmv(True)
    l0 = c.launch_count()
    c.profile_bytes(reset=True)
    barrier()
    c.profiler_range(True)
    c.timer_start()
    t0 = time.perf_counter()
    stats = [step(False) for _ in range(args.steps)]
    ms_dev = c.timer_stop()
    c.profiler_range(False)
    barrier()
    wall = time.perf_counter() - t0
    launches = c.launch_count() - l0
    step_bytes = c.profile_bytes()   # algorithmic bytes of every launch of the timed region, by kernel class (this rank)
    n_spmv, spmv_ms = c.profile_spmv_get()
    c.profile_spmv(False)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:   # before the end-to-end leg below overwrites u
        dump_outputs(args.dump_outputs, c.download(u, 3), stats[-1])
    # ---- end-to-end: same step through the C ABI with host buffers (H2D of u, D2H of the updated u) ----
    step(True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(True)
    barrier()
    wall_e2e = time.perf_counter() - t0
    # ---- the two flavours of jacobian_volume, one launch each on the step's state (outside the timed step): the step uses
    # the exact derivative; the reference's NumericalJacobianVolume replay (FD-faithful) is reported beside it ----
    A2 = c.matrix(h)
    jac_ms = {}
    for name_, mode_ in (("analytic", capi.JAC_ANALYTIC), ("fd_faithful", capi.JAC_FD_FAITHFUL)):
        c.jacobian(h, us, A2, mode_, 1e-11)
        barrier()
        c.timer_start(); c.jacobian(h, us, A2, mode_, 1e-11); jac_ms[name_] = c.timer_stop()
    c.matrix_destroy(A2)
    # ---- N > 1: the step's result against the 1-rank result of the same step ----
    parity = None
    if world > 1 and not args.no_check:
        step(False)
        parity = parity_vs_n1(args, c, capi, u, fine_plan, rank, world, dist, torch, cfg, a, jac_mode)
    tmax = torch.tensor([ms_dev / 1e3, wall, wall_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        sb = torch.tensor([step_bytes[k] for k in sorted(step_bytes)], dtype=torch.float64, device="cuda")
        dist.all_reduce(sb)
        step_bytes = dict(zip(sorted(step_bytes), [float(v) for v in sb.tolist()]))
    sec_dev, wall, wall_e2e = [float(v) for v in tmax.tolist()]
    sec_step = max(sec_dev, 0.0) / args.steps
    if rank != 0:
        return
    r = stats[-1]
    peak, peak_src = measured_peaks()
    # algorithmic bytes of one fine-level 3-field SpMV (DESIGN.md "SpMV"): 7 value planes + column index per
    # slot, row pointer + x read + y written per vertex
    # per epilogue kind: plain y = A x; residual and smoother step also read b (24 B/vertex).  The smoother's own x row is part
    # of the x read, and its 3x3 inverse diagonal block is computed in the kernel from the diagonal slot, not read.
    base = (7 * 8 + 4) * ns + (4 + 2 * 3 * 8) * n_own   # rank 0's share
    kind_bytes = [base, base + 24 * n_own, base + 24 * n_own]
    spmv_total_bytes = sum(b * n for b, n in zip(kind_bytes, n_spmv))
    spmv_ms_by_kind, n_spmv_by_kind = spmv_ms, n_spmv
    spmv_ms, n_spmv = sum(spmv_ms), sum(n_spmv)
    spmv_bytes = spmv_total_bytes / max(n_spmv, 1)
    spmv_avg_s = spmv_ms / 1e3 / max(n_spmv, 1)
    achieved = spmv_bytes / spmv_avg_s / 1e9
    asm_s = float(np.mean([x.seconds_assembly for x in stats]))
    cpu = None
    if not args.no_cpu:  # bounded CPU sample on all host cores (and the single-core phases beside it)
        from oracle import binding as ora
        nthr = args.cpu_threads if args.cpu_threads > 0 else ora.max_threads()
        lvl = args.cpu_level if args.cpu_level >= 0 else 5
        cpu = cpu_newton_step(lvl, nthr, krylov_iters=max(1, int(r.linear_iterations)))
        cpu1 = cpu_newton_step(lvl, 1, krylov_iters=1) if nthr > 1 else cpu
    line = {
        "metric": METRIC, "value": gdof / sec_step, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec_step * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "test/pore_pnp (pore.msh + pore.cfg) uniformly refined %d times: one monolithic PNP Newton "
                               "step (Jacobian assembly, BiCGSTAB + multigrid, line search)" % args.levels,
                   "levels": args.levels, "dofs": gdof, "matrix_slots": gslots,
                   "rank0_owned_vertices": n_own, "rank0_ghost_vertices": nv - n_own,
                   "parallelism": "1 GPU" if world == 1 else "%d subdomains (RCB of the Gmsh mesh, %s partitioner), NCCL halo exchange per multigrid level + scalar allreduce" % (world, "numpy" if PYTHON_PARTITIONER else "native"),
                   "jacobian": args.jac, "solver_options": dict(EXTRA_SOLVER_OPTS), "preconditioner": "multigrid V(%d,%d), damped Jacobi: %s" % (args.prec_steps, args.prec_steps,
                       "refinement levels with P1 interpolation + re-discretised operators, aggregation AMG below the Gmsh mesh" if world == 1
                       else "distributed refinement levels with P1 interpolation, re-discretised operators, " + ("replicated dense LU on the Gmsh mesh" if DENSE_COARSE else "levels <= %d replicated on every rank (one-GPU hierarchy: refinement levels, aggregation AMG below the Gmsh mesh)" % REPLICA_LEVEL)),
                   "start_state": "PNP solution of level %d, P1-interpolated" % args.coarse_level,
                   "l2_policy": "inputs larger than L2 (per GPU: matrix %.1f GB, vectors %.2f GB each)" % (7 * 8 * ns / 1e9, 8 * ndof / 1e9)},
        "newton_step_s": sec_step, "assembled_dofs_per_s": gdof / asm_s if asm_s > 0 else None,
        "jacobian_ms": jac_ms, "newton_step_s_with_fd_jacobian": sec_step + (jac_ms["fd_faithful"] - jac_ms["analytic"]) / 1e3,
        "krylov_iterations": int(r.linear_iterations), "line_search_trials": int(r.line_search_trials),
        "defect_before": r.first_defect, "defect_after": r.defect, "parity_vs_n1": parity,
        "spmv_gbs": achieved, "spmv_launches_timed": n_spmv,
        "spmv_by_kind": {k: {"launches": n, "avg_ms": (m / n if n else None), "bytes": b} for k, n, m, b in
                         zip(["plain", "residual", "smoother"], n_spmv_by_kind, spmv_ms_by_kind, kind_bytes)}, "spmv_share_of_step": spmv_ms / 1e3 / max(sec_dev, 1e-30),
        "setup_s": t_setup, "wall_s": wall,
        "roofline": {"bound": "hbm", "kernel": "3-field SpMV on the vertex-star layout, fine level (k_star_op_tma<7,EPI,NDOT,2>: bulk-copy "
                               "pipeline, all epilogues -- plain / dots, residual, smoother step)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     # DRAM bytes per launch from the committed `ncu --set full` capture of this kernel at this size (smoother
                     # epilogue, 59 % of the launches: 22.37 GB read + 1.13 GB written against 23.34 GB algorithmic; residual
                     # epilogue 22.41 + 1.13 GB); other sizes: not captured
                     "traffic": 23.50e9 if (world == 1 and args.levels == 7) else None,
                     "traffic_source": "ncu dram__bytes_read.sum + dram__bytes_write.sum of k_star_op_tma<7,2,0,2> at k = 7 "
                                       "(profiles/hot_kernels_full_r02_summary.txt); algorithmic bytes of that epilogue: 23.34e9",
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": spmv_bytes,  # launch-weighted mean over the epilogue kinds
                     "avg_launch_ms": spmv_avg_s * 1e3,
                     # the WHOLE step: algorithmic bytes of every kernel launched in the timed region (all ranks), by class,
                     # over the step time -- against the measured copy bandwidth and the nominal 8 TB/s of the north star
                     "step": {"bytes_per_step": sum(step_bytes.values()) / args.steps,
                              "by_class_gb": {k: v / args.steps / 1e9 for k, v in step_bytes.items()},
                              "achieved": sum(step_bytes.values()) / args.steps / sec_step / 1e9 / world, "unit": "GB/s per GPU",
                              "frac": sum(step_bytes.values()) / args.steps / sec_step / 1e9 / world / peak,
                              "frac_of_8000": sum(step_bytes.values()) / args.steps / sec_step / 1e9 / world / 8000.0}},
        "cpu_baseline": None if cpu is None else {
            "value": cpu["value"], "unit": UNIT, "cores": cpu["threads"], "kind": "port", "sample": cpu_sample_text(cpu),
            "phases_s": cpu["phases_s"], "assembled_dofs_per_s": cpu["assembled_dofs_per_s"], "spmv_gbs": cpu["spmv_gbs"],
            "single_core_phases_s": cpu1["phases_s"]},
        "e2e": {"value": gdof / (wall_e2e / args.steps), "unit": UNIT, "h2d_bytes_per_step": 8 * ndof * world,
                "d2h_bytes_per_step": 8 * ndof * world},
        "gpu_launches": int(launches), "clocks": clocks, "coarse_correction_cuda_graph": int(c.solver_get(s, "amg_graph")),
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--levels", type=int, default=7, help="uniform refinements of pore.msh (7 -> 141 M dofs)")
    ap.add_argument("--coarse-level", type=int, default=3)
    ap.add_argument("--cpu-level", type=int, default=-1, help="refinement level of the CPU arm (default: 5 -> 8.84 M dofs, BASELINE.md "
                    "section 4; --impl reference with more than 8 steps in all: 4, so that the run ends within a few minutes)")
    ap.add_argument("--cpu-threads", type=int, default=0, help="host threads of the CPU arm (0: all cores)")
    ap.add_argument("--prec-steps", type=int, default=2)
    ap.add_argument("--jac", choices=["analytic", "fd"], default="analytic")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="N > 1: skip parity_vs_n1 (rank 0 re-runs the step on one GPU and compares)")
    ap.add_argument("--solver-opt", action="append", default=[], metavar="NAME=VALUE",
                    help="pnp_solver_set_option for the timed step's multigrid (experiments), e.g. amg_smoother=1")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--replica-level", type=int, default=3, help="N > 1: levels below this one run replicated on every rank (no halo exchanges there)")
    ap.add_argument("--python-partitioner", action="store_true", help="N > 1: numpy partitioner (dune_pnp_b200/partition.py) instead of the native one")
    ap.add_argument("--dense-coarse", action="store_true", help="N > 1: replicated dense LU on the Gmsh mesh instead of the replica hierarchy")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's outputs to DIR/*.npy "
                    "(one GPU, b200 implementation)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs the b200 implementation on one GPU")
    global DENSE_COARSE, REPLICA_LEVEL, PYTHON_PARTITIONER
    DENSE_COARSE = args.dense_coarse; REPLICA_LEVEL = args.replica_level; PYTHON_PARTITIONER = args.python_partitioner
    for kv in args.solver_opt:
        k, v = kv.split("=")
        EXTRA_SOLVER_OPTS[k] = float(v)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_gpu(args, rank, world, local_rank)
        if world > 1:
            # every rank leaves together and at once: the line is out; finalisers of NCCL-backed objects (torch's process
            # group, the library's communicator, CUDA graphs holding NCCL nodes) have no defined order at interpreter exit
            import torch.distributed as dist
            try:
                dist.barrier()
            except Exception:
                pass
            sys.stdout.flush(); sys.stderr.flush()
            os._exit(0)


if __name__ == "__main__":
    main()
