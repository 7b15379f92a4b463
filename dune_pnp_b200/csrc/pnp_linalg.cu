// pnp_linalg.cu -- device Krylov stack: SpMV on the star layout, fused BLAS-1, BiCGSTAB and CG.
//
// Replaces ISTL's BiCGSTABSolver / CGSolver as wrapped by PDELab's ISTLBackend_NOVLP_* backends
// (/root/reference/src/instationary_pnp_from_pb_md.hh:188-211, stationary_pnp.hh:254-256); the
// iteration follows dune-istl 2.2 solvers.hh as restated in SURVEY.md App. A.7 (half-iteration
// counting, convergence tests after each half step, breakdown thresholds 1e-80).
//
// All kernels are HBM-bound.  SpMV bytes per launch: nplanes*8*nslots (values) + 4*nslots (adj)
// + 4*nv (rp) + 16*F*nv (x read once if the gather hits cache, y written).  Dot products ride in
// the epilogue of the kernel that produces their operand; reductions are two-stage and
// deterministic (per-block partials, then one block).
#include <chrono>
#include <cmath>

#include "pnp_common.cuh"
#include "pnp_spmv_tma.cuh"

namespace pnp {

namespace {

constexpr int RED_BLOCK = 256;
constexpr int MAX_RED = 4; // values reduced per launch

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// block-wide sums of NR values; result valid in thread 0, written to partial[blockIdx.x*NR + j]
template <int NR> __device__ __forceinline__ void block_partials(double (&v)[NR], double* __restrict__ partial) {
  __shared__ double sm[NR][RED_BLOCK / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < NR; j++) {
    double s = warp_sum(v[j]);
    if (lane == 0) sm[j][w] = s;
  }
  __syncthreads();
  if (w == 0) {
#pragma unroll
    for (int j = 0; j < NR; j++) {
      double s = lane < (blockDim.x >> 5) ? sm[j][lane] : 0.0;
      s = warp_sum(s);
      if (lane == 0) partial[(long)blockIdx.x * NR + j] = s;
    }
  }
}
__global__ void k_reduce_final(const double* __restrict__ partial, int nblocks, int nr, double* __restrict__ out) {
  __shared__ double sm[RED_BLOCK / 32];
  for (int j = 0; j < nr; j++) {
    double s = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += blockDim.x) s += partial[(long)i * nr + j];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
      double t = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.0;
      t = warp_sum(t);
      if (threadIdx.x == 0) out[j] = t;
    }
    __syncthreads();
  }
}

// ---- fused BLAS-1 ----
__global__ void __launch_bounds__(RED_BLOCK) k_dot(const double* __restrict__ a, const double* __restrict__ b, long n,
                                                   double* __restrict__ partial) {
  double s[1] = {0.0};
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) s[0] += a[i] * b[i];
  block_partials<1>(s, partial);
}
// r = b - t (residual from a product); partial: |r|^2
__global__ void __launch_bounds__(RED_BLOCK) k_sub_norm(const double* b, const double* __restrict__ t, double* r, long n,
                                                        double* __restrict__ partial) { // b may alias r
  double s[1] = {0.0};
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const double v = b[i] - t[i];
    r[i] = v; s[0] += v * v;
  }
  block_partials<1>(s, partial);
}
// x += a*y ; r -= a*v ; partial: |r|^2 and rt.r
__global__ void __launch_bounds__(RED_BLOCK)
k_update_xr(double a, const double* __restrict__ y, const double* __restrict__ v, double* __restrict__ x,
            double* __restrict__ r, const double* __restrict__ rt, long n, double* __restrict__ partial) {
  double s[2] = {0.0, 0.0};
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    x[i] += a * y[i];
    const double ri = r[i] - a * v[i];
    r[i] = ri; s[0] += ri * ri; s[1] += rt[i] * ri;
  }
  block_partials<2>(s, partial);
}
// p = r + beta*(p - omega*v)   (ISTL: p.axpy(-omega,v); p *= beta; p += r)
__global__ void k_update_p(double beta, double omega, const double* __restrict__ r, const double* __restrict__ v,
                           double* __restrict__ p, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    p[i] = (p[i] - omega * v[i]) * beta + r[i];
}
__global__ void k_axpy(double a, const double* __restrict__ x, double* __restrict__ y, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) y[i] += a * x[i];
}
// p = beta*p + q
__global__ void k_xpby(double beta, const double* __restrict__ q, double* __restrict__ p, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) p[i] = beta * p[i] + q[i];
}
__global__ void k_set(double* __restrict__ x, long n, double v) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) x[i] = v;
}
// Jacobi: inverse of the scalar diagonal (ISTLBackend_NOVLP_CG_Jacobi, SURVEY App. A.8)
template <int NP>
__global__ void k_diag_inverse(const int* __restrict__ rp, const double* __restrict__ vals, long stride, int nv,
                               double* __restrict__ dinv) {
  constexpr int F = NP == 1 ? 1 : 3;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    const int s = rp[v];
    if (NP == 1) dinv[v] = 1.0 / vals[s];
    else {
      const PnpBlock B = pnp_block_at<NP>(vals, stride, s);
      dinv[(long)F * v] = 1.0 / B.a;
      dinv[(long)F * v + 1] = 1.0 / B.e;
      dinv[(long)F * v + 2] = 1.0 / B.g;
    }
  }
}
// y = dinv .* d ; optionally partial: y.d   (CG's rho = (q,b))
template <int NDOT>
__global__ void __launch_bounds__(RED_BLOCK) k_diag_apply(const double* __restrict__ dinv, const double* __restrict__ d,
                                                          double* __restrict__ y, long n, double* __restrict__ partial) {
  double s[1] = {0.0};
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const double v = dinv[i] * d[i];
    y[i] = v; s[0] += v * d[i];
  }
  if (NDOT) block_partials<1>(s, partial);
}

int red_grid(const Ctx& c, long n) { return grid_for(n, RED_BLOCK, c.sm_count * 4); }

void ensure_red(Ctx& c) {
  const size_t need = (size_t)c.sm_count * 8 * MAX_RED;
  if (c.red_partial.n < need) c.red_partial.alloc(need);
  if (c.red_out.n < MAX_RED) c.red_out.alloc(MAX_RED);
  if (!c.h_red) PNP_CUDA(cudaMallocHost(&c.h_red, MAX_RED * sizeof(double)));
}
// second stage + readback of nr values produced by `nblocks` blocks
void finish_reduce(Ctx& c, int nblocks, int nr, double* out) {
  k_reduce_final<<<1, RED_BLOCK, 0, c.stream>>>(c.red_partial.p, nblocks, nr, c.red_out.p);
  PNP_CHECK_LAUNCH(); c.launches++;
  allreduce_sum(c, c.red_out.p, nr); // sum over ranks (no-op on one GPU)
  PNP_CUDA(cudaMemcpyAsync(c.h_red, c.red_out.p, nr * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  for (int j = 0; j < nr; j++) out[j] = c.h_red[j];
}

// y = A x with optional fused dots; returns them in dots[0..ndot)
void spmv_dots(Ctx& c, const Matrix& A, double* x, double* y, int ndot, const double* w1, double* dots) {
  ensure_red(c);
  PNP_REQUIRE(c.degree == 1 || A.csr_rp, PNP_E_ARG, "matrix not assembled (or detached by a parameter change): assemble it first");
  if (A.csr_rp) { // quadratic elements: CSR rows, the dots as separate reductions
    csr_spmv(c, A, x, y);
    if (ndot >= 1) dots[0] = vec_dot(c, y, w1, A.csr_n);
    if (ndot == 2) dots[1] = vec_dot(c, y, y, A.csr_n);
    return;
  }
  halo_exchange(c, x, A.nplanes == 1 ? 1 : 3); // ghost columns of x (no-op on one GPU)
  StarOpArgs a{c.rp.p, c.adj.p, A.vals.p, c.nslots, (int)c.n_own, x, y};
  a.w1 = w1; a.partial = c.red_partial.p;
  c.prof_mark();
  const int grid = ndot == 0 ? launch_star_op_auto<EPI_PLAIN, 0>(c, A.nplanes, a)
                 : ndot == 1 ? launch_star_op_auto<EPI_PLAIN, 1>(c, A.nplanes, a) : launch_star_op_auto<EPI_PLAIN, 2>(c, A.nplanes, a);
  c.prof_mark();
  if (ndot > 0) finish_reduce(c, grid, ndot, dots);
}

} // namespace

void spmv(Ctx& c, const Matrix& A, double* x, double* y) { spmv_dots(c, A, x, y, 0, nullptr, nullptr); }

double vec_dot(Ctx& c, const double* x, const double* y, long n) {
  ensure_red(c);
  const int g = red_grid(c, n);
  k_dot<<<g, RED_BLOCK, 0, c.stream>>>(x, y, n, c.red_partial.p);
  PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, (x == y ? 8.0 : 16.0) * n);
  double d;
  finish_reduce(c, g, 1, &d);
  return d;
}
double vec_norm(Ctx& c, const double* x, long n) { return std::sqrt(vec_dot(c, x, x, n)); }
void vec_axpy(Ctx& c, double a, const double* x, double* y, long n) {
  k_axpy<<<grid_for(n, 256), 256, 0, c.stream>>>(a, x, y, n);
  PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 24.0 * n);
}
void vec_copy(Ctx& c, const double* x, double* y, long n) {
  PNP_CUDA(cudaMemcpyAsync(y, x, n * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
  c.acct(Ctx::ACC_BLAS1, 16.0 * n);
}
void vec_zero(Ctx& c, double* x, long n) { PNP_CUDA(cudaMemsetAsync(x, 0, n * sizeof(double), c.stream)); c.acct(Ctx::ACC_BLAS1, 8.0 * n); }

// ---- preconditioner dispatch ----------------------------------------------------------------
void amg_setup(Ctx&, Solver&, const Matrix&);                        // pnp_amg.cu
void amg_apply(Ctx&, Solver&, const Matrix&, const double* d, double* y); // pnp_amg.cu
void ssor_setup(Ctx&, Solver&, const Matrix&);                       // pnp_precond.cu
void ssor_apply(Ctx&, Solver&, const Matrix&, const double* d, double* y);
void ilu0_setup(Ctx&, Solver&, const Matrix&);
void ilu0_apply(Ctx&, Solver&, const Matrix&, const double* d, double* y);

namespace {
void prec_setup(Ctx& c, Solver& S, const Matrix& A) {
  PNP_REQUIRE(c.degree == 1 || A.csr_rp, PNP_E_ARG, "matrix not assembled (or detached by a parameter change): assemble it first");
  if (A.csr_rp) {
    if (S.prec == PNP_PREC_AMG) pmg_setup(c, S, A);
    if (S.prec == PNP_PREC_JACOBI) csr_diag_inverse(c, A, S.dinv.p);
    if (S.prec == PNP_PREC_SSOR || S.prec == PNP_PREC_ILU0) csr_sweep_setup(c, S, A, S.prec == PNP_PREC_ILU0);
    return;
  }
  switch (S.prec) {
    case PNP_PREC_NONE: break;
    case PNP_PREC_JACOBI: {
      const int g = grid_for(c.n_own, 256);
      if (A.nplanes == 1) k_diag_inverse<1><<<g, 256, 0, c.stream>>>(c.rp.p, A.vals.p, c.nslots, (int)c.n_own, S.dinv.p);
      else if (A.nplanes == PNP_COMPACT_PLANES)
        k_diag_inverse<PNP_COMPACT_PLANES><<<g, 256, 0, c.stream>>>(c.rp.p, A.vals.p, c.nslots, (int)c.n_own, S.dinv.p);
      else k_diag_inverse<7><<<g, 256, 0, c.stream>>>(c.rp.p, A.vals.p, c.nslots, (int)c.n_own, S.dinv.p);
      PNP_CHECK_LAUNCH(); c.launches++;
      break;
    }
    case PNP_PREC_SSOR: ssor_setup(c, S, A); break;
    case PNP_PREC_ILU0: ilu0_setup(c, S, A); break;
    case PNP_PREC_AMG: amg_setup(c, S, A); break;
    default: PNP_REQUIRE(false, PNP_E_ARG, "unknown preconditioner");
  }
}
// y = M^{-1} d  (ISTL: y = 0; prec.apply(y, d))
void prec_apply(Ctx& c, Solver& S, const Matrix& A, const double* d, double* y, long n) {
  switch (S.prec) {
    case PNP_PREC_NONE: vec_copy(c, d, y, n); break; // Richardson: y = d
    case PNP_PREC_JACOBI:
      k_diag_apply<0><<<grid_for(n, RED_BLOCK), RED_BLOCK, 0, c.stream>>>(S.dinv.p, d, y, n, nullptr);
      PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 24.0 * n);
      break;
    case PNP_PREC_SSOR: if (A.csr_rp) csr_ssor_apply(c, S, A, d, y); else ssor_apply(c, S, A, d, y); break;
    case PNP_PREC_ILU0: if (A.csr_rp) csr_ilu0_apply(c, S, A, d, y); else ilu0_apply(c, S, A, d, y); break;
    case PNP_PREC_AMG: if (A.csr_rp) pmg_apply(c, S, A, d, y); else amg_apply(c, S, A, d, y); break;
    default: break;
  }
}

LinResult finish(LinResult res, double it, double norm, double norm0, bool conv, int status) {
  res.converged = conv; res.status = status;
  res.iterations = (int)std::ceil(it);
  res.reduction = norm0 > 0 ? norm / norm0 : 0.0;
  res.conv_rate = it > 0 ? std::pow(res.reduction, 1.0 / it) : 0.0;
  return res;
}

// BiCGSTABSolver::apply(x, b): b is overwritten with the residual (SURVEY App. A.7)
LinResult bicgstab(Ctx& c, Solver& S, const Matrix& A, double* x, double* r, long n, double reduction) {
  LinResult res;
  double *rt = S.w[0].p, *p = S.w[1].p, *v = S.w[2].p, *t = S.w[3].p, *y = S.w[4].p;
  double red[MAX_RED];
  const int g = red_grid(c, n);
  // r = b - A x
  spmv(c, A, x, t);
  k_sub_norm<<<g, RED_BLOCK, 0, c.stream>>>(r, t, r, n, c.red_partial.p);
  PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 24.0 * n);
  finish_reduce(c, g, 1, red);
  vec_copy(c, r, rt, n);
  vec_zero(c, p, n); vec_zero(c, v, n);
  double rho = 1, alpha = 1, omega = 1, rho_new, beta, h;
  const double norm0 = std::sqrt(red[0]);
  double norm = norm0;
  double it = 0;
  if (!std::isfinite(norm0)) return finish(res, it, norm, norm0, false, PNP_E_NAN);
  if (norm < reduction * norm0 || norm < 1e-30) return finish(res, it, norm, norm0, true, 0);
  rho_new = red[0]; // rt = r  =>  (rt, r) = |r|^2
  for (it = 0.5; it < S.maxit; it += 0.5) {
    if (std::fabs(rho) <= 1e-80 || std::fabs(omega) <= 1e-80) return finish(res, it, norm, norm0, false, PNP_E_BREAKDOWN);
    if (it < 1) vec_copy(c, r, p, n);
    else {
      beta = (rho_new / rho) * (alpha / omega);
      k_update_p<<<grid_for(n, 256), 256, 0, c.stream>>>(beta, omega, r, v, p, n);
      PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 32.0 * n);
    }
    prec_apply(c, S, A, p, y, n);
    spmv_dots(c, A, y, v, 1, rt, red); // v = A y ; h = (rt, v)
    h = red[0];
    if (std::fabs(h) < 1e-80 || !std::isfinite(h)) return finish(res, it, norm, norm0, false, PNP_E_BREAKDOWN);
    alpha = rho_new / h;
    k_update_xr<<<g, RED_BLOCK, 0, c.stream>>>(alpha, y, v, x, r, rt, n, c.red_partial.p);
    PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 56.0 * n);
    finish_reduce(c, g, 2, red);
    norm = std::sqrt(red[0]);
    if (S.verbosity > 1) std::printf("  BiCGSTAB %5.1f  %.6e\n", it, norm);
    if (norm < reduction * norm0) return finish(res, it, norm, norm0, true, 0);
    it += 0.5;
    prec_apply(c, S, A, r, y, n);
    spmv_dots(c, A, y, t, 2, r, red); // t = A y ; (t, r), (t, t)
    omega = red[0] / red[1];
    k_update_xr<<<g, RED_BLOCK, 0, c.stream>>>(omega, y, t, x, r, rt, n, c.red_partial.p);
    PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 56.0 * n);
    finish_reduce(c, g, 2, red);
    rho = rho_new;
    norm = std::sqrt(red[0]);
    rho_new = red[1]; // (rt, r) for the next half step, fused into the update
    if (S.verbosity > 1) std::printf("  BiCGSTAB %5.1f  %.6e\n", it, norm);
    if (!std::isfinite(norm)) return finish(res, it, norm, norm0, false, PNP_E_NAN);
    if (norm < reduction * norm0 || norm < 1e-30) return finish(res, it, norm, norm0, true, 0);
  }
  return finish(res, S.maxit, norm, norm0, false, 0);
}

// CGSolver::apply(x, b)
LinResult cg(Ctx& c, Solver& S, const Matrix& A, double* x, double* b, long n, double reduction) {
  LinResult res;
  double *p = S.w[0].p, *q = S.w[1].p;
  double red[MAX_RED];
  const int g = red_grid(c, n);
  spmv(c, A, x, q);
  k_sub_norm<<<g, RED_BLOCK, 0, c.stream>>>(b, q, b, n, c.red_partial.p);
  PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 24.0 * n);
  finish_reduce(c, g, 1, red);
  const double def0 = std::sqrt(red[0]);
  double def = def0;
  int i = 0;
  if (!std::isfinite(def0)) return finish(res, 0, def, def0, false, PNP_E_NAN);
  if (def0 < 1e-30) return finish(res, 0, def, def0, true, 0);
  prec_apply(c, S, A, b, p, n);
  double rholast = vec_dot(c, p, b, n);
  for (i = 1; i <= S.maxit; i++) {
    spmv_dots(c, A, p, q, 1, p, red); // q = A p ; alpha = (p, q)
    const double lambda = rholast / red[0];
    k_update_xr<<<g, RED_BLOCK, 0, c.stream>>>(lambda, p, q, x, b, p, n, c.red_partial.p);
    PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 56.0 * n);
    finish_reduce(c, g, 2, red);
    def = std::sqrt(red[0]);
    if (S.verbosity > 1) std::printf("  CG %5d  %.6e\n", i, def);
    if (!std::isfinite(def)) return finish(res, i, def, def0, false, PNP_E_NAN);
    if (def < def0 * reduction || def < 1e-30) return finish(res, i, def, def0, true, 0);
    prec_apply(c, S, A, b, q, n);
    const double rho = vec_dot(c, q, b, n);
    const double beta = rho / rholast;
    k_xpby<<<grid_for(n, 256), 256, 0, c.stream>>>(beta, q, p, n);
    PNP_CHECK_LAUNCH(); c.launches++; c.acct(Ctx::ACC_BLAS1, 24.0 * n);
    rholast = rho;
  }
  return finish(res, S.maxit, def, def0, false, 0);
}
} // namespace

void precond_apply(Ctx& c, Solver& S, const Matrix& A, Vec& d, Vec& v) {
  PNP_REQUIRE(d.fields == v.fields && d.fields == (A.nplanes == 1 ? 1 : 3) && d.d.p != v.d.p, PNP_E_ARG,
              "vector field count does not match the matrix");
  S.ensure((size_t)c.cols() * d.fields);
  ensure_red(c);
  prec_setup(c, S, A);
  prec_apply(c, S, A, d.d.p, v.d.p, c.rows() * d.fields);
}

LinResult solver_apply(Ctx& c, Solver& S, const Matrix& A, Vec& z, Vec& r, double reduction) {
  PNP_REQUIRE(z.fields == r.fields && z.fields == (A.nplanes == 1 ? 1 : 3), PNP_E_ARG,
              "vector field count does not match the matrix");
  const long n = c.rows() * z.fields; // owned dofs: what dots, norms and updates run over
  S.ensure((size_t)c.cols() * z.fields);  // work vectors carry a ghost part for the SpMV input
  ensure_red(c);
  auto t0 = std::chrono::steady_clock::now();
  prec_setup(c, S, A);
  LinResult res = S.kind == PNP_SOLVER_CG ? cg(c, S, A, z.d.p, r.d.p, n, reduction)
                                          : bicgstab(c, S, A, z.d.p, r.d.p, n, reduction);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  res.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return res;
}

} // namespace pnp
