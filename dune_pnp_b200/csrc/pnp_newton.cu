// pnp_newton.cu -- Dune::PDELab::Newton and StationaryLinearProblemSolver on the device.
//
// Flow restated from PDELab 1.1 newton.hh / linearproblem.hh (SURVEY.md App. A.1, A.9) as the
// reference drives them: /root/reference/src/stationary_pnp_from_pb.hh:172-185 (PB) and :344-360
// (PNP); instationary_pnp_from_pb_md.hh:214-228, :349-350.  u, z, r, the trial iterates of the
// Hackbusch-Reusken line search and the matrix stay in HBM; only the scalar defect norms and the
// Krylov scalars reach the host.
#include <chrono>
#include <cmath>

#include "pnp_common.cuh"

namespace pnp {

// Value planes of a PNP Jacobian of this context (pnp_jacobian_planes of its parameter set): the compact layout needs one
// unpartitioned GPU mesh.
int pnp_context_planes(const Ctx& c, int jac_mode, bool solver_ok) {
  if (c.n_own != c.nv || !c.mg.empty()) return op_planes(OP_PNP);
  std::vector<int> btype;
  for (const HostSurface& s : c.params.surfaces) btype.insert(btype.end(), s.btype, s.btype + 3);
  return pnp_jacobian_planes(jac_mode, c.degree, solver_ok, btype.data(), (int)c.params.surfaces.size());
}

namespace {
double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// Value planes of the work-space Jacobian: the compact PNP layout (pnp_jacobian_planes) where the solver reads the matrix
// through star SpMVs and diagonal blocks only -- no preconditioner, Jacobi, or the multigrid with the Jacobi or Chebyshev
// smoother -- on one GPU.  Everything else keeps the operator's planes.
int workspace_planes(const Ctx& c, const Operator& op, const Solver& S, int jac_mode) {
  if (op.op != OP_PNP || !tune().jac_compact) return op_planes(op.op);
  const double sm = S.opt("amg_smoother", 0);
  const bool solver_ok = S.prec == PNP_PREC_NONE || S.prec == PNP_PREC_JACOBI || (S.prec == PNP_PREC_AMG && (sm == 0 || sm == 1));
  return pnp_context_planes(c, jac_mode, solver_ok);
}
} // namespace

int newton_apply(Ctx& c, const Operator& op, Vec& u, Solver& S, const pnp_newton_opts& o, pnp_newton_result& R) {
  const int F = op_fields(op.op);
  PNP_REQUIRE(u.fields == F, PNP_E_ARG, "vector field count does not match the operator");
  const long n = c.rows() * F, nall = c.cols() * F;
  R = pnp_newton_result();
  Vec &r = c.ws_r, &z = c.ws_z, &prev_u = c.ws_prev;
  Matrix& A = c.ws_A;
  r.fields = z.fields = prev_u.fields = F;
  if (r.d.n != (size_t)nall) { r.d.alloc(nall); z.d.alloc(nall); prev_u.d.alloc(nall); }
  r.d.zero(c.stream); z.d.zero(c.stream);
  A.op = op.op; A.nplanes = workspace_planes(c, op, S, o.jac_mode);
  if (c.degree >= 2) p2_matrix_init(c, A, op);
  else if (A.vals.n != (size_t)A.nplanes * c.nslots) A.vals.alloc((size_t)A.nplanes * c.nslots);
  const double t_start = now();
  auto sync = [&] { PNP_CUDA(cudaStreamSynchronize(c.stream)); };
  auto defect = [&]() {
    const double t0 = now();
    assemble_residual(c, op, u, r);
    const double d = vec_norm(c, r.d.p, n);
    R.seconds_assembly += now() - t0;
    R.residual_assemblies++;
    return d;
  };
  auto record = [&](double d, int lin_its) {
    if (R.n_history < 64) { R.defect_history[R.n_history] = d; R.linear_iterations_history[R.n_history] = lin_its; R.n_history++; }
  };
  int status = PNP_OK;
  R.defect = defect();
  R.first_defect = R.defect;
  double prev_defect = R.defect;
  // PDELab's Newton sets reassemble_threshold = 0 after a line-search failure on a matrix that was not reassembled
  // (newton.hh, NewtonLineSearchError handler): the next pass is forced to assemble, whatever the threshold says
  double reassemble_threshold = o.reassemble_threshold;
  int ls_retries = 0;
  record(R.defect, 0);
  if (!std::isfinite(R.defect)) { R.seconds_total = now() - t_start; return PNP_E_NAN; }
  if (o.verbosity >= 2) std::printf("  Initial defect: %12.4e\n", R.defect);
  while (true) {
    R.converged = R.defect < o.abs_limit || R.defect < R.first_defect * o.reduction;
    if (R.converged) break;
    if (R.iterations >= o.max_iterations) { status = PNP_E_NOT_CONVERGED; break; }
    // prepare_step
    bool reassembled = false;
    if (R.defect / prev_defect > reassemble_threshold || R.jacobian_assemblies == 0) {
      const double t0 = now();
      assemble_jacobian(c, op, u, A, o.jac_mode, o.fd_epsilon);
      sync();
      R.seconds_assembly += now() - t0;
      R.jacobian_assemblies++;
      reassembled = true;
    }
    const double stop_defect = std::max(R.first_defect * o.reduction, o.abs_limit);
    const double ratio2 = R.defect * R.defect / (prev_defect * prev_defect);
    const double linear_reduction =
        stop_defect / (10 * R.defect) > ratio2 ? stop_defect / (10 * R.defect) : std::min(o.min_linear_reduction, ratio2);
    prev_defect = R.defect;
    // linearSolve
    vec_zero(c, z.d.p, n);
    const double t1 = now();
    const LinResult lr = solver_apply(c, S, A, z, r, linear_reduction);
    R.seconds_solve += now() - t1;
    R.linear_iterations += lr.iterations;
    if (o.verbosity >= 3)
      std::printf("  linear solve: %d its, reduction %.3e (asked %.3e)\n", lr.iterations, lr.reduction, linear_reduction);
    if (!lr.converged) {
      record(R.defect, lr.iterations);
      status = lr.status == PNP_E_BREAKDOWN ? PNP_E_BREAKDOWN : PNP_E_LINEAR_SOLVER;
      break;
    }
    // line_search: hackbuschReuskenAcceptBest (the reference drivers' choice), hackbuschReusken or noLineSearch
    double lambda = 1.0, best_lambda = 0.0, best_defect = R.defect;
    vec_copy(c, u.d.p, prev_u.d.p, n);
    int i = 0;
    bool ls_failed = false;
    while (true) {
      vec_axpy(c, -lambda, z.d.p, u.d.p, n);
      R.defect = defect();
      R.line_search_trials++;
      if (o.line_search_strategy == PNP_LS_NONE) break; // noLineSearch: the full step is taken whatever the defect does
      const bool finite = std::isfinite(R.defect);
      if (finite && R.defect <= (1.0 - lambda / 4) * prev_defect) break;
      if (finite && R.defect < best_defect) { best_defect = R.defect; best_lambda = lambda; }
      if (++i >= o.line_search_max_iterations) {
        if (best_lambda == 0.0 || o.line_search_strategy == PNP_LS_HACKBUSCH_REUSKEN) {
          vec_copy(c, prev_u.d.p, u.d.p, n);
          R.defect = defect();
          ls_failed = true;
          break;
        }
        if (best_lambda != lambda) {
          vec_copy(c, prev_u.d.p, u.d.p, n);
          vec_axpy(c, -best_lambda, z.d.p, u.d.p, n);
          R.defect = defect();
        }
        break;
      }
      lambda *= o.damping;
      vec_copy(c, prev_u.d.p, u.d.p, n);
    }
    if (ls_failed) {
      // a retry is only worth it with a freshly assembled matrix, and only once per step (bounded loop)
      if (reassembled || ++ls_retries > o.max_iterations) { status = PNP_E_LINE_SEARCH; break; }
      reassemble_threshold = 0.0; // defect / prev_defect is exactly 1 now: forces the assembly
      continue;
    }
    reassemble_threshold = o.reassemble_threshold;
    R.reduction = R.defect / R.first_defect;
    R.iterations++;
    record(R.defect, lr.iterations);
    if (o.verbosity >= 2)
      std::printf("  Newton iteration %2d.  New defect: %12.4e.  Reduction (total): %12.4e  lambda %g  lin its %d\n",
                  R.iterations, R.defect, R.reduction, lambda, lr.iterations);
  }
  sync();
  R.seconds_total = now() - t_start;
  return status;
}

// StationaryLinearProblemSolver::apply: A = J(u); r = R(u); solve A z = r to `reduction`; u -= z
LinResult slp_apply(Ctx& c, const Operator& op, Vec& u, Solver& S, double reduction, int jac_mode, double eps) {
  const int F = op_fields(op.op);
  PNP_REQUIRE(u.fields == F, PNP_E_ARG, "vector field count does not match the operator");
  const long n = c.rows() * F, nall = c.cols() * F;
  Vec &r = c.ws_r, &z = c.ws_z;
  Matrix& A = c.ws_A;
  r.fields = z.fields = F;
  if (r.d.n != (size_t)nall) { r.d.alloc(nall); z.d.alloc(nall); c.ws_prev.d.alloc(nall); }
  r.d.zero(c.stream); z.d.zero(c.stream);
  A.op = op.op; A.nplanes = workspace_planes(c, op, S, jac_mode);
  if (c.degree >= 2) p2_matrix_init(c, A, op);
  else if (A.vals.n != (size_t)A.nplanes * c.nslots) A.vals.alloc((size_t)A.nplanes * c.nslots);
  assemble_jacobian(c, op, u, A, jac_mode, eps);
  assemble_residual(c, op, u, r);
  vec_zero(c, z.d.p, n);
  LinResult lr = solver_apply(c, S, A, z, r, reduction);
  // an ISTL breakdown throws before the update in the reference: u stays untouched
  if (lr.status != PNP_E_BREAKDOWN && lr.status != PNP_E_NAN) vec_axpy(c, -1.0, z.d.p, u.d.p, n);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  return lr;
}

// ---- OneStepMethod + OneStepGridOperator (SURVEY App. A.9; /root/reference/src/instationary_pnp_from_pb_md.hh:368-391,
// applied per time step at :421-425) ------------------------------------------------------------------------------
namespace {
struct TimeMethod { int s; double d[3], a[2][3], b[2][3]; };
TimeMethod time_method(int method) {
  if (method == PNP_TIME_IMPLICIT_EULER) return TimeMethod{1, {0.0, 1.0, 0.0}, {{-1.0, 1.0, 0.0}, {0, 0, 0}}, {{0.0, 1.0, 0.0}, {0, 0, 0}}};
  PNP_REQUIRE(method == PNP_TIME_ALEXANDER2, PNP_E_ARG, "unknown time stepping method");
  const double al = 1.0 - 0.5 * std::sqrt(2.0); // Alexander2Parameter
  return TimeMethod{2, {0.0, al, 1.0}, {{-1.0, 1.0, 0.0}, {-1.0, 0.0, 1.0}}, {{0.0, al, 0.0}, {0.0, 1.0 - al, al}}};
}
// A = a*A + b*B over all slots
__global__ void k_stage_matrix(double* __restrict__ A, const double* __restrict__ B, double a, double b, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) A[i] = a * A[i] + b * B[i];
}
// constrained rows of the combined matrix are trivial: unit diagonal (their off-diagonals are zero in both parts)
__global__ void k_unit_dirichlet_diag(const int* __restrict__ rp, const unsigned char* __restrict__ dmask, int comp, int n_own,
                                      double* __restrict__ A) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n_own; v += gridDim.x * blockDim.x)
    if ((dmask[v] >> comp) & 1u) A[rp[v]] = 1.0;
}
// Dirichlet dofs take the boundary function's values (interpolate + copy_nonconstrained_dofs)
__global__ void k_set_dirichlet(const unsigned char* __restrict__ dmask, int comp, int n, const double* __restrict__ g,
                                double* __restrict__ x) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x)
    if ((dmask[v] >> comp) & 1u) x[v] = g[v];
}
// y = (init ? 0 : y) + a*p + b*q
__global__ void k_lincomb(double* __restrict__ y, int init, double a, const double* __restrict__ p, double b,
                          const double* __restrict__ q, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    double v = init ? 0.0 : y[i];
    if (p) v += a * p[i];
    if (q) v += b * q[i];
    y[i] = v;
  }
}
} // namespace

// xold -> xnew over one step dt.  op0: spatial operator (GO0), op1: temporal operator (GO1); g: Dirichlet values; each
// stage is one StationaryLinearProblemSolver::apply on  a_rr*M + b_rr*dt*J0.  stage[r] receives the stage solves' results.
int onestep_apply(Ctx& c, int method, const Operator& op0, const Operator& op1, Solver& S, double dt, Vec& xold, Vec& g,
                  Vec& xnew, double reduction, int jac_mode, double eps, LinResult* stage) {
  PNP_REQUIRE(op_fields(op0.op) == 1 && op_fields(op1.op) == 1, PNP_E_ARG, "one-step method: scalar operators expected");
  PNP_REQUIRE(xold.fields == 1 && xnew.fields == 1 && g.fields == 1, PNP_E_ARG, "one-step method: 1-field vectors expected");
  PNP_REQUIRE(op0.comp0 == op1.comp0, PNP_E_ARG, "spatial and temporal operator must share the constraints");
  const TimeMethod tm = time_method(method);
  const long n = c.rows(), nall = c.cols();
  const int comp = op0.comp0;
  const bool p2 = c.degree >= 2;
  for (auto& v : c.ws_stage) { v.fields = 1; if (v.d.n != (size_t)nall) { v.d.alloc(nall); v.d.zero(c.stream); } }
  Vec &x1 = c.ws_stage[0], &x2 = c.ws_stage[1], &cst = c.ws_stage[2], &r0 = c.ws_stage[3], &r1 = c.ws_stage[4];
  Vec &r = c.ws_r, &z = c.ws_z;
  r.fields = z.fields = 1;
  if (r.d.n != (size_t)nall) { r.d.alloc(nall); z.d.alloc(nall); c.ws_prev.d.alloc(nall); r.d.zero(c.stream); z.d.zero(c.stream); }
  Matrix &A = c.ws_A, &B = c.ws_B;
  A.op = op0.op; B.op = op1.op; A.nplanes = B.nplanes = 1;
  if (p2) { p2_matrix_init(c, A, op0); p2_matrix_init(c, B, op1); }
  else {
    if (A.vals.n != (size_t)c.nslots) A.vals.alloc(c.nslots);
    if (B.vals.n != (size_t)c.nslots) B.vals.alloc(c.nslots);
  }
  const long nvals = p2 ? A.csr_nnz : c.nslots;
  Vec* x[3] = {&xold, &x1, &x2};
  const int gv = grid_for(n, 256), gs = grid_for(nvals, 256);
  for (int rs = 1; rs <= tm.s; rs++) {
    // preStage: the part of the stage residual that the earlier stages fix
    bool first = true;
    for (int i = 0; i < rs; i++) {
      const double ai = tm.a[rs - 1][i], bi = tm.b[rs - 1][i];
      const bool do1 = std::fabs(ai) > 1e-6, do0 = std::fabs(bi) > 1e-6;
      if (do1) assemble_residual(c, op1, *x[i], r1);
      if (do0) assemble_residual(c, op0, *x[i], r0);
      if (do0 || do1) {
        k_lincomb<<<gv, 256, 0, c.stream>>>(cst.d.p, first, ai, do1 ? r1.d.p : nullptr, bi * dt, do0 ? r0.d.p : nullptr, n);
        PNP_CHECK_LAUNCH(); c.launches++;
        first = false;
      }
    }
    if (first) vec_zero(c, cst.d.p, n);
    Vec& xn = *x[rs];
    vec_copy(c, x[rs - 1]->d.p, xn.d.p, n);
    k_set_dirichlet<<<gv, 256, 0, c.stream>>>(p2 ? p2_dirichlet_flags(c) : c.dmask.p, comp, (int)n, g.d.p, xn.d.p);
    PNP_CHECK_LAUNCH(); c.launches++;
    const double ar = tm.a[rs - 1][rs], br = tm.b[rs - 1][rs];
    assemble_jacobian(c, op1, xn, B, jac_mode, eps);
    assemble_jacobian(c, op0, xn, A, jac_mode, eps);
    k_stage_matrix<<<gs, 256, 0, c.stream>>>(A.vals.p, B.vals.p, br * dt, ar, nvals);
    // (a constrained CSR row holds its diagonal alone, a constrained star row starts with it)
    k_unit_dirichlet_diag<<<gv, 256, 0, c.stream>>>(p2 ? A.csr_rp : c.rp.p, p2 ? p2_dirichlet_flags(c) : c.dmask.p, comp, (int)n, A.vals.p);
    PNP_CHECK_LAUNCH(); c.launches += 2;
    c.last_vals = nullptr; // A is a combination now: a multigrid must not re-discretise `op0` for it
    assemble_residual(c, op1, xn, r1);
    assemble_residual(c, op0, xn, r0);
    vec_copy(c, cst.d.p, r.d.p, n);
    k_lincomb<<<gv, 256, 0, c.stream>>>(r.d.p, 0, ar, r1.d.p, br * dt, r0.d.p, n);
    PNP_CHECK_LAUNCH(); c.launches++;
    vec_zero(c, z.d.p, n);
    const LinResult lr = solver_apply(c, S, A, z, r, reduction);
    if (stage) stage[rs - 1] = lr;
    if (lr.status) return lr.status;
    vec_axpy(c, -1.0, z.d.p, xn.d.p, n);
  }
  vec_copy(c, x[tm.s]->d.p, xnew.d.p, n);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  return 0;
}

} // namespace pnp
