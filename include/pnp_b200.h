/* pnp_b200.h -- C ABI of the B200 backend for dune-pnp's Newton-step hot path.
 *
 * The reference (/root/reference, a DUNE/PDELab application) has no FFI: its drivers call C++
 * templates of PDELab/ISTL directly.  Each entry point below names the reference call it stands in
 * for (paths relative to /root/reference/src); INTEGRATION.md shows the PDELab-shaped C++ facade
 * (include/pnp_b200/pdelab_facade.hh) a maintainer binds instead of the upstream templates.
 *
 * Conventions
 *  - every function returns a pnp_status; the message of the last failure is pnp_last_error(ctx);
 *    no C++ exception crosses this boundary.
 *  - host arrays are copied; device memory is owned by the context; vectors/matrices/operators/
 *    solvers are small integer handles valid for the life of the context.
 *  - the numbering seen through this header is the reference's: vertex index = rank of the Gmsh node
 *    id among nodes used by triangles (GmshReader), P1 dof = vertex index, 3-field dof =
 *    field*nv + vertex (GridFunctionSpaceLexicographicMapper, stationary_pnp.hh:126-129).
 *    Internally vertices are renumbered for locality and dofs are vertex-blocked.
 *  - one context drives one GPU; calls are synchronous; a context is not re-entrant.
 */
#ifndef PNP_B200_H
#define PNP_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pnp_ctx pnp_ctx;
typedef int pnp_status;

enum {
  PNP_OK = 0,
  PNP_E_NOT_CONVERGED = 1, /* Dune::PDELab::NewtonNotConverged */
  PNP_E_LINEAR_SOLVER = 2, /* NewtonLinearSolverError */
  PNP_E_LINE_SEARCH = 3,   /* NewtonLineSearchError */
  PNP_E_NAN = 4,           /* NewtonDefectError */
  PNP_E_BREAKDOWN = 5,     /* Dune::ISTLError (BiCGSTAB rho/omega/h breakdown) */
  PNP_E_CUDA = 6,
  PNP_E_CONFIG = 7,        /* missing INI key / unreadable file (sysparams.cc:24-28) */
  PNP_E_ARG = 8,
  PNP_E_MESH = 9           /* degenerate / non-manifold / too large mesh */
};

/* local operators (files of the same name under /root/reference/src) */
enum { PNP_OP_PB = 0, PNP_OP_POISSON = 1, PNP_OP_DIFFUSION = 2, PNP_OP_MASS = 3, PNP_OP_PNP = 4 };
/* jacobian_volume flavour: the reference inherits NumericalJacobianVolume (pnp_operator.hh:24-27) */
enum { PNP_JAC_FD_FAITHFUL = 0, PNP_JAC_ANALYTIC = 1 };
/* ISTLBackend_NOVLP_* solver/preconditioner pairs (instationary_pnp_from_pb_md.hh:188-211) */
enum { PNP_SOLVER_BCGS = 0, PNP_SOLVER_CG = 1 };
enum { PNP_PREC_NONE = 0, PNP_PREC_JACOBI = 1, PNP_PREC_SSOR = 2, PNP_PREC_ILU0 = 3, PNP_PREC_AMG = 4 };

/* ---- context ------------------------------------------------------------------------------ */
pnp_status pnp_ctx_create(int device, pnp_ctx** out);
void pnp_ctx_destroy(pnp_ctx* ctx);
const char* pnp_last_error(pnp_ctx* ctx);
/* process-wide kernel tuning knobs (experiments, tests): "tma" (1: large levels run the bulk-copy streaming SpMV, 0: the
 * plain-load kernel everywhere), "tma_stages" (2..3), "tma_min_rows" (smallest level served by the streaming kernel, -1:
 * two tiles per SM), "tma_lpr" (lanes per row, 1 or 2), "mg_f32_min_rows" (smallest multigrid level whose damped-Jacobi
 * smoother and residual read a single-precision copy of the level's matrix -- one GPU, levels the streaming kernel
 * serves; -1: 2^22 rows, 1: every such level, a huge value: none), "graph" (1: the multigrid's coarse correction is
 * replayed from a CUDA graph), "matrix_compact" (1: pnp_matrix_create gives PNP matrices the compact 5-plane layout where the exact
 * Jacobian has it -- linear elements, every surface constraining all three fields or none, one unpartitioned mesh;
 * pnp_matrix_set_csr, FD assembly, SSOR, ILU0 and the Gauss-Seidel smoother refuse such a matrix) */
pnp_status pnp_tune(const char* name, double value);
/* number of CUDA kernels this context has launched so far */
long pnp_launch_count(pnp_ctx* ctx);

/* measurement hooks (bench.py): CUDA events on the context's stream.  pnp_profile_spmv(ctx,1) brackets every
 * fine-level SpMV launch with an event pair; pnp_profile_spmv_get() returns their count and summed duration. */
pnp_status pnp_profile_spmv(pnp_ctx*, int enable);
/* launches[3], total_ms[3]: by epilogue kind -- 0: y = A x (+ fused dots), 1: y = b - A x, 2: smoother step */
pnp_status pnp_profile_spmv_get(pnp_ctx*, long* launches, double* total_ms);
/* ALGORITHMIC bytes (compulsory traffic: every array a kernel must read or write, once) of all launches since the last
 * reset, by kernel class: out6 = {fine-level SpMV, coarser-level SpMV, assembly (residual, Jacobian, coarse operators),
 * vector updates / reductions / copies, grid transfers (restriction, prolongation, first smoothing step), dense coarse solve} */
pnp_status pnp_profile_bytes(pnp_ctx*, int reset, double* out6);
/* cudaProfilerStart/Stop: lets `ncu --profile-from-start off` see only the timed region */
pnp_status pnp_profiler_range(pnp_ctx*, int start);
pnp_status pnp_timer_start(pnp_ctx*);
pnp_status pnp_timer_stop(pnp_ctx*, double* elapsed_ms);

/* ---- mesh: GmshReader<UGGrid<2>>::read + createGrid (pnp_solver_main.cc:82-114) ---------- */
pnp_status pnp_mesh_set(pnp_ctx*, long nv, const double* x, const double* y, long nT, const int* tri /*[nT][3]*/,
                        long nB, const int* ba, const int* bb, const int* bphys);
pnp_status pnp_mesh_read_gmsh(pnp_ctx*, const char* path);
/* ---- multi-GPU: one context per rank owns a subdomain (replaces grid->loadBalance(), pnp_solver_main.cc:108, and the
 * PDELab "nonoverlapping" machinery: GridOperator<...,true>, NonoverlappingOperator/ScalarProduct, stationary_pnp.hh:240).
 * Local mesh: the first n_own vertices are owned (they get matrix rows), the rest are ghosts grouped by owner rank; all
 * elements touching an owned vertex must be present.  pnp_halo_set(): per neighbour rank i, send_idx[send_ptr[i]:
 * send_ptr[i+1]] are the owned local vertices whose values that rank needs, and the ghosts [n_own + recv_ptr[i],
 * n_own + recv_ptr[i+1]) are received from it in the order that rank sends them.  NCCL carries only these halo values
 * and the scalar sums of dot products / norms. */
pnp_status pnp_mesh_set_local(pnp_ctx*, long nv, long n_own, const double* x, const double* y, long nT, const int* tri,
                              long nB, const int* ba, const int* bb, const int* bphys);
pnp_status pnp_mesh_owned(pnp_ctx*, long* n_own);
pnp_status pnp_comm_unique_id(char* out128);                 /* ncclGetUniqueId on rank 0, broadcast by the launcher */
pnp_status pnp_comm_init(pnp_ctx*, int rank, int world, const char* unique_id128);
/* the same with the id passed through a file every rank can see (a C++ driver started by any process launcher, no MPI):
 * rank 0 writes it, the others wait for it */
pnp_status pnp_comm_init_file(pnp_ctx*, int rank, int world, const char* path);
/* all-gather of byte blocks of different lengths over the context's communicator (set-up plumbing: the two exchanges of
 * pnp_part_*): counts[world]; recv == NULL: sizes only */
pnp_status pnp_comm_allgatherv(pnp_ctx*, const void* send, long nbytes, void* recv, long cap, long* counts);
pnp_status pnp_halo_set(pnp_ctx*, int n_nbr, const int* nbr, const int* send_ptr, const int* send_idx, const int* recv_ptr);
pnp_status pnp_halo_exchange(pnp_ctx*, int vec_handle);       /* refresh the ghost part of a vector */
/* distributed geometric multigrid: a child context (same stream and communicator) holds this rank's part of a coarser
 * mesh level (pnp_mesh_set_local + pnp_halo_set + pnp_mesh_finalize on the child).  pnp_mg_push_level registers it as the
 * next coarser level: par0/par1[v] = parents of local vertex v of the next finer level (caller's local numbering on both
 * levels, -1: none; one parent: coinciding vertex, two: midpoint of a coarse edge).  Coarse operators are re-discretised
 * on the child meshes; the coarsest level is gathered by its global vertex indices and solved redundantly by dense LU. */
pnp_status pnp_ctx_create_child(pnp_ctx* parent, pnp_ctx** child);
pnp_status pnp_mg_push_level(pnp_ctx*, pnp_ctx* child, const int* par0, const int* par1);
pnp_status pnp_mg_set_coarse_global(pnp_ctx*, const int* global_vertex_index, long n_global);
/* alternative: the coarsest pushed level stays a smoothed level and the dense system is its Galerkin aggregate:
 * aggregate[v] = aggregate index of local vertex v (the same global aggregation on every rank) */
pnp_status pnp_mg_set_coarse_aggregates(pnp_ctx*, const int* aggregate, long n_aggregates);
/* third variant: `replica` is a child context that holds the WHOLE coarsest mesh on every rank (pnp_mesh_set +
 * pnp_mesh_finalize on the child; global_vertex_index[v] = replica vertex of local vertex v of the coarsest pushed
 * level).  The coarsest distributed level is then gathered to the replica (allreduce of F values per vertex) and the
 * replica runs the single-GPU multigrid below it (aggregation levels, small dense LU) redundantly on every rank: the
 * cycle equals the one-GPU cycle, and no rank factorises a matrix of the size of the coarsest mesh. */
pnp_status pnp_mg_set_coarse_replica(pnp_ctx*, pnp_ctx* replica, const int* global_vertex_index, long n_global);
/* ---- native domain decomposition: grid->loadBalance() (pnp_solver_main.cc:93-108) --------------------------------------
 * Host code, no GPU needed.  Every rank calls pnp_part_create with the SAME coarse mesh: recursive coordinate bisection of
 * the triangle centroids into `world` parts, this rank's part with one ghost layer, `levels` uniform refinements of that
 * local mesh (trimmed back to one layer after each).  Per level, coarsest first, the halo plan needs two small all-gathers
 * whose transport is the caller's (MPI in a DUNE build, torch.distributed in the Python launchers, pnp_comm_allgatherv):
 *   pnp_part_ghost_keys  -> (x bits, y bits) of this rank's ghost vertices            [all-gather: every rank's keys]
 *   pnp_part_claim       -> for every rank q the positions of q's ghosts owned here    [all-gather: every rank's claims]
 *   pnp_part_finalize    <- the positions of MY ghosts each rank r claimed (mine_ptr[r] .. mine_ptr[r+1])
 * after which pnp_part_sizes / pnp_part_get return the level in the form pnp_mesh_set_local / pnp_halo_set /
 * pnp_mg_push_level take: owned vertices first, ghosts grouped by owner rank in the order the owner sends them; par0/par1 =
 * parents in the next coarser level's numbering; gid (coarsest level) = global vertex index.
 * sizes[8] = {nv, n_own, nT, nB, n_nbr, n_send, n_global, has_gid}. */
typedef struct pnp_part pnp_part;
pnp_status pnp_part_create(long nv, const double* x, const double* y, long nT, const int* tri, long nB, const int* ba,
                           const int* bb, const int* bphys, int world, int rank, int levels, pnp_part** out);
void pnp_part_destroy(pnp_part*);
const char* pnp_part_last_error(pnp_part*);
pnp_status pnp_part_ghost_keys(pnp_part*, int level, long* n, unsigned long long* keys /* 2*n, may be NULL */);
pnp_status pnp_part_claim(pnp_part*, int level, const long* ghost_ptr /* world+1 */, const unsigned long long* ghost_keys_all,
                          long* claim_ptr /* world+1 */, long* claim_pos /* may be NULL */);
pnp_status pnp_part_finalize(pnp_part*, int level, const long* mine_ptr /* world+1 */, const long* mine_pos);
pnp_status pnp_part_sizes(pnp_part*, int level, long* sizes);
pnp_status pnp_part_get(pnp_part*, int level, double* x, double* y, int* tri, int* ba, int* bb, int* bphys, int* nbr,
                        int* send_ptr, int* send_idx, int* recv_ptr, int* par0, int* par1, int* gid);
/* The whole decomposition in one call (a driver without a Python launcher: PnpSolverMain::run with N ranks).  `root` holds
 * the GLOBAL coarse mesh, the parameters and an initialised communicator on every rank; afterwards it holds this rank's part
 * of the mesh refined `levels` times, the coarser levels are its multigrid levels down to `replica_level`, and a replica of the
 * whole mesh continues below on every rank.  The level contexts belong to root.  Optional nodal fields given on the
 * unpartitioned mesh of refinement level `field_level` (values [nfields][nf] at vertices (fx, fy)[nf], e.g. a coarse solution)
 * are injected there by coordinate match and P1-interpolated to the finest level into a new vector *start_vec. */
pnp_status pnp_partition_build(pnp_ctx* root, int levels, int replica_level, int field_level, int nfields, long nf,
                               const double* fx, const double* fy, const double* fields, int* start_vec);
/* uniform red refinement on the device (synthetic large meshes; rule in DESIGN.md) */
pnp_status pnp_mesh_refine(pnp_ctx*, int levels);
/* nested iteration: pnp_carry_set() stores vectors in reference numbering; every later pnp_mesh_refine() level
 * interpolates them (P1: midpoint average) to the finer mesh; after pnp_mesh_finalize() they are read back with
 * pnp_carry_get() into freshly created vectors.  Setting or refining a mesh invalidates all vector, matrix,
 * operator and solver handles. */
pnp_status pnp_carry_set(pnp_ctx*, const int* vec_handles, int n);
pnp_status pnp_carry_get(pnp_ctx*, int index, int vec_handle);
/* same, for a field given / returned in reference numbering on the host ([fields][nv]); needs no finalized mesh */
pnp_status pnp_carry_set_host(pnp_ctx*, int fields, const double* host);
pnp_status pnp_carry_get_host(pnp_ctx*, int index, double* host);
/* dof_perm hook: new_index[v] = the caller's index of vertex v (a bijection).  The numbering at this boundary is the
 * numbering of the mesh arrays; a caller whose grid numbers the vertices differently from the Gmsh file (UGGrid's leaf
 * index after loadBalance(), pnp_solver_main.cc:106-114) renumbers a mesh read with pnp_mesh_read_gmsh before finalizing
 * it, and from then on vectors, patterns, matrices, constraints and sweep orders follow the caller's numbering. */
pnp_status pnp_mesh_renumber(pnp_ctx*, const int* new_index);
/* builds the vertex-star structure; renumber != 0 reorders vertices internally for locality */
pnp_status pnp_mesh_finalize(pnp_ctx*, int renumber);
pnp_status pnp_mesh_sizes(pnp_ctx*, long* nv, long* nT, long* nB, long* nslots);
pnp_status pnp_mesh_get(pnp_ctx*, double* x, double* y, int* tri, int* ba, int* bb, int* bphys);

/* ---- parameters: Sysparams::readConfigFile (sysparams.cc:15-98) --------------------------- */
/* sys[16] = {n_surfaces, cylindrical, l_b, c0, PI, linearSolverIterations, newtonReassembleThreshold,
 *            newtonReduction, newtonMinLinearReduction, newtonMaxIterations,
 *            newtonLineSearchMaxIteration, tau, nSteps, outputFreq, potentialUpdateFreq, verbosity}
 * surf[n_surfaces][9] = per BC component {coulomb, plusDiffusion, minusDiffusion}: {Btype, Flux, Dirichlet value} */
pnp_status pnp_params_set(pnp_ctx*, const double* sys, const double* surf);
pnp_status pnp_params_read(pnp_ctx*, const char* cfg_path);
pnp_status pnp_params_get(pnp_ctx*, double* sys, double* surf /* may be NULL */, char* meshfile, int meshfile_cap);
/* constraints(bctype, gfs, cc) for all three BC components at once (btype.hh:21-53; stationary_pnp.hh:155) */
pnp_status pnp_constraints_build(pnp_ctx*);

/* ---- operators: LocalOperator + GridOperator (stationary_pnp.hh:218-241) ------------------ */
/* comp0: BC component the scalar operator's BCType was instantiated with (ignored for PNP) */
pnp_status pnp_operator_create(pnp_ctx*, int op, int comp0, int* op_handle);
/* coefficient grid functions: Poisson which=0:c+ 1:c- (poisson_operator.hh:97-100); diffusion which=0: Phi */
pnp_status pnp_operator_set_coefficient(pnp_ctx*, int op_handle, int which, int vec_handle);
pnp_status pnp_operator_set_valency(pnp_ctx*, int op_handle, double valency);
/* Dirichlet flags per dof, reference numbering */
pnp_status pnp_constraints_get(pnp_ctx*, int op_handle, char* is_dirichlet);
/* MatrixContainer pattern (ISTLBCRSMatrixBackend<1,1>): rows ascending, columns ascending, constrained rows
 * reduced to the diagonal.  col == NULL: only *nnz (and rowptr if given) is produced. */
pnp_status pnp_pattern_get(pnp_ctx*, int op_handle, long* nnz, int* rowptr, int* col);

/* ---- vectors: ISTLVectorBackend<1> containers --------------------------------------------- */
pnp_status pnp_vec_create(pnp_ctx*, int fields, int* vec_handle);
pnp_status pnp_vec_destroy(pnp_ctx*, int vec_handle);
pnp_status pnp_vec_upload(pnp_ctx*, int vec_handle, const double* host);
pnp_status pnp_vec_download(pnp_ctx*, int vec_handle, double* host);
pnp_status pnp_vec_set(pnp_ctx*, int vec_handle, double value);
pnp_status pnp_vec_copy(pnp_ctx*, int dst, int src);
pnp_status pnp_vec_axpy(pnp_ctx*, int y, double a, int x); /* y += a x */
pnp_status pnp_vec_norm(pnp_ctx*, int x, double* two_norm);
pnp_status pnp_vec_dot(pnp_ctx*, int x, int y, double* result);

/* ---- assembly: GridOperator::residual / ::jacobian (stationary_pnp.hh:240-246) ------------ */
pnp_status pnp_matrix_create(pnp_ctx*, int op_handle, int* mat_handle);
pnp_status pnp_matrix_destroy(pnp_ctx*, int mat_handle);
pnp_status pnp_residual(pnp_ctx*, int op_handle, int u, int r);
pnp_status pnp_jacobian(pnp_ctx*, int op_handle, int u, int mat_handle, int mode, double fd_epsilon);
/* values in the order of pnp_pattern_get() */
pnp_status pnp_matrix_values_get(pnp_ctx*, int op_handle, int mat_handle, double* val);
pnp_status pnp_spmv(pnp_ctx*, int mat_handle, int x, int y);
/* the ISTL-backend-level drop-in: values of an EXTERNALLY assembled matrix in the container layout of pnp_pattern_get()
 * -- what A.base() of the ISTLBCRSMatrixBackend<1,1> matrix holds when the driver calls ls.apply(A, z, r, red)
 * (instationary_pnp_from_pb_md.hh:188-211; stationary_pnp.hh:247).  rowptr / col must equal the operator's pattern; a
 * multigrid preconditioner treats such a matrix with Galerkin coarse operators. */
pnp_status pnp_matrix_set_csr(pnp_ctx*, int op_handle, int mat_handle, const int* rowptr, const int* col, const double* val);

/* ---- linear solvers: ISTLBackend_NOVLP_*::apply / result (instationary_pnp_from_pb_md.hh:188-211) */
typedef struct {
  int converged;
  int iterations;
  double reduction;
  double conv_rate;
  double seconds;
  int status;
} pnp_lin_result;
pnp_status pnp_solver_create(pnp_ctx*, int kind, int prec, int maxit, int prec_steps, int verbosity, int* solver);
/* tuning knobs of the preconditioner, by name: "amg_smoother" (0 damped Jacobi, 1 Chebyshev), "amg_omega",
 * "amg_alpha" (coarse-correction scaling, dune-istl default 1.6), "amg_gamma" (1 V-cycle, 2 W-cycle), "amg_wlevels" (W on the first n levels only),
 * "amg_coarse_sweeps", "amg_dense_max" (coarsest level with at most this many dofs is solved by dense LU; 0: sweeps),
 * "amg_cheb_ratio" (lambda_max / lambda_min of the Chebyshev interval), "amg_pre_steps" / "amg_post_steps" (smoothing
 * steps before / after the coarse correction; default: the solver's prec_steps for both), "amg_geometric" (default 1: when
 * the mesh was refined with pnp_mesh_refine, the coarser refinement levels become multigrid levels with P1
 * interpolation; aggregation continues below the coarsest mesh), "amg_rediscretise" (default 1: the operators of those
 * levels are re-discretised on the level meshes at the injected state when the matrix is the Jacobian of the last
 * pnp_jacobian / Newton assembly of a PB, PNP or mass operator; 0 or any other matrix: Galerkin products) */
pnp_status pnp_solver_set_option(pnp_ctx*, int solver, const char* name, double value);
/* read-back of solver facts, by name: "ssor_levels" / "ilu0_levels" (number of levels of the level-scheduled sweep that
 * reproduces SeqSSOR / SeqILU0 in the reference's row order; 0 before the first use), "amg_graph" (1: the multigrid's coarse
 * correction runs from a CUDA graph, -1: capture was not possible, 0: not captured yet) */
pnp_status pnp_solver_get(pnp_ctx*, int solver, const char* name, double* value);
/* one application of the solver's preconditioner, v = M^-1 d, as ISTL's Preconditioner::pre/apply/post on the matrix
 * (SeqSSOR / SeqILU0 / SeqJac / AMG / Richardson).  d and v are distinct vectors of the matrix' field count. */
pnp_status pnp_precond_apply(pnp_ctx*, int solver, int mat_handle, int d, int v);
/* z: initial guess in, solution out; r: right-hand side in, residual out (as ISTL does) */
pnp_status pnp_solver_apply(pnp_ctx*, int solver, int mat_handle, int z, int r, double reduction, pnp_lin_result*);

/* ---- Newton: Dune::PDELab::Newton (stationary_pnp.hh:280-294) ------------------------------ */
/* Newton::setLineSearchStrategy (stationary_pnp.hh:283): PDELab 1.1's three strategies */
enum { PNP_LS_HACKBUSCH_REUSKEN_ACCEPT_BEST = 0, PNP_LS_NONE = 1, PNP_LS_HACKBUSCH_REUSKEN = 2 };
typedef struct {
  double reduction;             /* setReduction */
  double abs_limit;             /* PDELab default 1e-12 */
  double min_linear_reduction;  /* setMinLinearReduction */
  double reassemble_threshold;  /* setReassembleThreshold */
  int max_iterations;           /* setMaxIterations */
  int line_search_max_iterations; /* setLineSearchMaxIterations */
  double damping;               /* 0.5 */
  int jac_mode;                 /* PNP_JAC_* */
  double fd_epsilon;            /* NumericalJacobianVolume epsilon: 1e-11 (PDELab <= 1.1) */
  int verbosity;
  int line_search_strategy;     /* setLineSearchStrategy: PNP_LS_* (the reference drivers pass hackbuschReuskenAcceptBest) */
} pnp_newton_opts;
typedef struct {
  int converged;
  int iterations;
  double first_defect, defect, reduction;
  int linear_iterations, line_search_trials, jacobian_assemblies, residual_assemblies;
  double seconds_assembly, seconds_solve, seconds_total;
  int n_history;
  double defect_history[64];
  int linear_iterations_history[64];
} pnp_newton_result;
void pnp_newton_opts_default(pnp_newton_opts*);
/* fills opts as the reference drivers do from Sysparams (stationary_pnp_from_pb.hh:344-351) */
pnp_status pnp_newton_opts_from_params(pnp_ctx*, pnp_newton_opts*);
pnp_status pnp_newton_apply(pnp_ctx*, int op_handle, int u, int solver, const pnp_newton_opts*, pnp_newton_result*);
/* StationaryLinearProblemSolver::apply (instationary_pnp_from_pb_md.hh:349-350) */
pnp_status pnp_slp_apply(pnp_ctx*, int op_handle, int u, int solver, double reduction, int jac_mode, double fd_epsilon,
                         pnp_lin_result*);

/* ---- time stepping: Dune::PDELab::OneStepMethod<Real,IGO,PDESOLVER,U,U>::apply(time, dt, xold, f, xnew) on a
 * OneStepGridOperator<GO0,GO1> with a StationaryLinearProblemSolver per stage (instationary_pnp_from_pb_md.hh:368-391,
 * applied at :421-425).  op_space = GO0's local operator (DiffusionOperator), op_time = GO1's (DiffusionTOperator);
 * dirichlet_values = the boundary function f interpolated to the dofs (only constrained dofs are read; the reference's
 * cpB/cmB are time independent); stage_results: one entry per stage (2 for Alexander2) or NULL. */
enum { PNP_TIME_ALEXANDER2 = 0, PNP_TIME_IMPLICIT_EULER = 1 };
pnp_status pnp_onestep_apply(pnp_ctx*, int method, int op_space, int op_time, int solver, double time, double dt, int x_old,
                             int dirichlet_values, int x_new, double reduction, int jac_mode, double fd_epsilon,
                             pnp_lin_result* stage_results);

/* ---- diagnostics of the time loop (instationary_pnp_from_pb_md.hh:430-452) --------------------------------- */
/* calcIonFlux (ionFlux.hh:8-96): ip[s], im[s] = currents of the two species through surface s, s < n_surfaces; the
 * reference appends "time ip[0] im[0] ip[1] im[1] ..." to current.dat.  With several ranks the sums run over all ranks. */
pnp_status pnp_ion_flux(pnp_ctx*, int phi, int cp, int cm, double* ip, double* im);
/* DataWriter::writeData (datawriter.hh:45-94): one text line per element, "x y<TAB>value<TAB>gradx grady", scientific
 * with precision 5, in grid element order */
pnp_status pnp_write_cell_data(pnp_ctx*, int vec_handle, const char* filename);

/* Dune::VTKWriter<GV>(gv, VTKOptions::conforming) + addVertexData(VTKGridFunctionAdapter(dgf, name)) + write(name,
 * VTKOptions::binaryappended) (instationary_pnp_from_pb_md.hh:337-340, :440; stationary_pnp_from_pb.hh:190-192, :386-390):
 * "<name>.vtu" with the n 1-field vectors as Float32 vertex data; ascii != 0: VTKOptions::ascii.  Several ranks: every
 * rank writes its piece "s<world>:p<rank>:<name>.vtu", rank 0 the "s<world>:<name>.pvtu" index. */
pnp_status pnp_write_vtk(pnp_ctx*, const char* name, int n, const int* vec_handles, const char* const* names, int ascii);

/* ---- initial guess / Dirichlet values: interpolate(BCExtension) (dirichlet_bc.hh:54-123) --- */
/* component 0: phi, 1: c+, 2: c-; pb_vec < 0 means a zero PB field; out is a 1-field vector */
pnp_status pnp_interpolate_bcext(pnp_ctx*, int component, int pb_vec, int out_vec);

/* ---- quadratic and cubic elements: the reference's -DPDEGREE=2 / -DPDEGREE=3 programs (src/Makefile.am:54-110;
 * Pk2DLocalFiniteElementMap<..., PDEGREE>, instationary_pnp_from_pb_md.hh:26-28,125; stationary_pnp.hh:190-193) ----
 * pnp_space_set_degree(ctx, 2 | 3) before pnp_mesh_finalize() selects the Pk space.  Scalar dofs per field, codim by codim
 * (SURVEY A.4): degree 3 first one bubble per element [0, nT); then degree-1 dofs per edge from `edge_offset` (edges ordered
 * by (min vertex, max vertex), pnp_space_edges; the dofs of an edge counted from its smaller end vertex); then one per vertex
 * from `vertex_offset`; fields lexicographic.  Vectors (pnp_vec_upload/download), constraints, patterns (pnp_pattern_get:
 * scalar BCRS, ascending columns) and matrix values use that numbering; it is also the device layout (CSR matrices, no
 * renumbering).  Operators, residual, Jacobian (both modes), SpMV, BiCGSTAB/CG with Richardson, Jacobi, SSOR(n) or ILU0
 * (row-order sweeps, level-scheduled), Newton, StationaryLinearProblemSolver, the one-step methods,
 * interpolate(BCExtension), calcIonFlux, writeData and the VTK vertex data work as for degree 1.  PNP_PREC_AMG is a
 * p-multigrid (SSOR on the Pk matrix, coarse correction in the P1 space through the multigrid of the linear-element path) for
 * the scalar operators on the last assembled Jacobian; the 3-field system, refinement carry-over and partitioned meshes answer
 * PNP_E_ARG.  One GPU. */
pnp_status pnp_space_set_degree(pnp_ctx*, int degree);
/* degree, number of edges (0 for degree 1) and scalar dofs per field */
pnp_status pnp_space_sizes(pnp_ctx*, int* degree, long* n_edges, long* ndof);
pnp_status pnp_space_edges(pnp_ctx*, int* va /*[n_edges]*/, int* vb);
/* first edge dof and first vertex dof of a field's block (degree 2: 0, n_edges; degree 3: nT, nT + 2 n_edges) */
pnp_status pnp_space_offsets(pnp_ctx*, long* edge_offset, long* vertex_offset);
/* Quadrature order of an operator (the `intorder` constructor argument, pb_operator.hh:39, pnp_operator.hh:40, ...).
 * 0 = what the reference's drivers end up with (3; DiffusionOperator 2; DiffusionTOperator 5), whatever PDEGREE is: with
 * cubic elements that rule under-integrates the element integrals and -- its centre weight being negative -- makes the PB / PNP
 * matrices indefinite (tests/test_oracle_p2.py); 5 (degree 2 and 3 only) selects the 7-point triangle rule and the 3-point
 * Gauss rule on faces, as passing intorder = 5 to the reference's constructors would. */
pnp_status pnp_operator_set_intorder(pnp_ctx*, int op_handle, int intorder);
/* packs three 1-field vectors into a 3-field vector / extracts one field */
pnp_status pnp_vec_pack3(pnp_ctx*, int dst3, int phi, int cp, int cm);
pnp_status pnp_vec_extract(pnp_ctx*, int src3, int field, int dst1);

#ifdef __cplusplus
}
#endif
#endif
