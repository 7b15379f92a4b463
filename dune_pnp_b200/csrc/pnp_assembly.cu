// pnp_assembly.cu -- residual and Jacobian assembly kernels (fp64, vertex-parallel gather).
//
// Replaces GridOperator::residual / GridOperator::jacobian driving the reference's local operators
// (/root/reference/src/stationary_pnp.hh:240-246; instationary_pnp_from_pb_md.hh:183-186,343-366):
// one thread owns one vertex row, walks the vertex star, recomputes the incident element integrals
// for its own test function and writes each result exactly once.  HBM-bound: per vertex it streams
// the ring (4 B/slot), gathers coordinates and coefficients (L1/L2 hits after the locality
// renumbering) and writes F residual entries or NPLANES*rowlen matrix values.
//
// This source is compiled TWICE (Makefile): with -DPNP_ASM_FAITHFUL -fmad=false it provides the FD-faithful Jacobian
// kernels, which must round like the CPU restatement (no FMA contraction, the reference's operation order); without
// the macro (FMA allowed) it provides the residual and exact-derivative Jacobian kernels plus the host-side dispatch.
#include "pnp_common.cuh"

namespace pnp {

// implemented in the other compilation of this file
void launch_jacobian_fd(Ctx& c, const StarView& M, const Operator& op, const double* u, const double* a0, const double* a1,
                        double* vals, long stride, double eps);

namespace {

// One block assembles the rows of 128 consecutive vertices per pass.  Their slots form ONE contiguous range of every
// value plane, so the rows are first written into a shared-memory tile (a thread's row is 7 doubles per plane: stored
// straight to global memory every store instruction of a warp touches 32 different sectors, and L2 evicts them half
// written -- the first version of this kernel read 15.7 GB and wrote 27.2 GB for an 18.4 GB matrix) and then copied out
// with fully coalesced stores.  Chunks with more than JAC_CAP slots (average valence > 8) are written directly.
constexpr int JAC_CHUNK = 128;   // = block size
constexpr int JAC_CAP = 1152;    // staged slots per plane

template <int OP, int MODE, int NP>
__global__ void __launch_bounds__(JAC_CHUNK)
k_jacobian(StarView M, PhysParams P, const double* __restrict__ u, const double* __restrict__ aux0,
           const double* __restrict__ aux1, double eps, int comp0, double* __restrict__ vals, long stride) {
  extern __shared__ double stage[]; // NP * JAC_CAP
  const int nchunks = (M.nv + JAC_CHUNK - 1) / JAC_CHUNK;
  for (int ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int v0 = ch * JAC_CHUNK, v1 = min(v0 + JAC_CHUNK, M.nv);
    const int sb = M.rp[v0], n = M.rp[v1] - sb;
    const int v = v0 + threadIdx.x;
    if (n <= JAC_CAP) { // block-uniform
      if (v < v1) jacobian_row<OP, MODE, NP>(M, P, u, aux0, aux1, eps, comp0, v, stage, JAC_CAP, sb);
      __syncthreads();
#pragma unroll
      for (int p = 0; p < NP; p++)
        for (int i = threadIdx.x; i < n; i += JAC_CHUNK) vals[p * stride + sb + i] = stage[p * JAC_CAP + i];
      __syncthreads();
    } else if (v < v1) {
      jacobian_row<OP, MODE, NP>(M, P, u, aux0, aux1, eps, comp0, v, vals, stride);
    }
  }
}

// M: the star to assemble on -- the context's own (finest) one, or a coarser refinement level's (multigrid)
template <int OP, int MODE, int NP = OpTraits<OP>::NPLANES>
void launch_jac(Ctx& c, const StarView& M, const Operator& op, const double* u, const double* a0, const double* a1,
                double* vals, long stride, double eps) {
  const PhysParams P = c.phys(op.valency);
  const int smem = NP * JAC_CAP * (int)sizeof(double);
  // (set on every launch: the attribute is per device and a process may drive several contexts)
  PNP_CUDA(cudaFuncSetAttribute(k_jacobian<OP, MODE, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int grid = grid_for(M.nv, JAC_CHUNK, c.sm_count * 16);
  k_jacobian<OP, MODE, NP><<<grid, JAC_CHUNK, smem, c.stream>>>(M, P, u, a0, a1, eps, op.comp0, vals, stride);
  PNP_CHECK_LAUNCH(); c.launches++;
  // ring (4 B/slot), row pointer + coordinates + Dirichlet mask + state (+ coefficient fields) per vertex, NP planes written
  c.acct(Ctx::ACC_ASSEMBLY, (4.0 + 8.0 * NP) * (double)stride + (21.0 + 8.0 * OpTraits<OP>::F + 8.0 * OpTraits<OP>::NAUX) * (double)M.nv);
}
// nplanes: the layout of the target matrix (the compact PNP layout is assembled by the exact derivative only)
template <int MODE>
void dispatch_jac(Ctx& c, const StarView& M, const Operator& op, const double* u, const double* a0, const double* a1,
                  double* vals, long stride, double eps, int nplanes) {
  if constexpr (MODE == JAC_ANALYTIC) {
    if (op.op == OP_PNP && nplanes == PNP_COMPACT_PLANES) {
      launch_jac<OP_PNP, JAC_ANALYTIC, PNP_COMPACT_PLANES>(c, M, op, u, a0, a1, vals, stride, eps);
      return;
    }
  }
  switch (op.op) {
    case OP_PB: launch_jac<OP_PB, MODE>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_POISSON: launch_jac<OP_POISSON, MODE>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_DIFFUSION: launch_jac<OP_DIFFUSION, MODE>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_MASS: launch_jac<OP_MASS, MODE>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_PNP: launch_jac<OP_PNP, MODE>(c, M, op, u, a0, a1, vals, stride, eps); break;
    default: PNP_REQUIRE(false, PNP_E_ARG, "unknown operator");
  }
}


// ---- NumericalJacobianVolume, warp-cooperative (the reference's own jacobian_volume: pnp_operator.hh:24-27, SURVEY A.3) ----
// The one-thread-per-vertex form above replays, for each of a vertex's ~6 elements, 1 + 3F residual evaluations in sequence
// at 255 registers and 8 warps per SM (134 ms for the 141 M-dof PNP matrix: 2.5 % of the HBM roofline, VERDICT r1).  Here a
// WARP owns the vertex and a LANE owns one evaluation: lane (g, c) evaluates ring element 3r + g with local dof c perturbed
// (c = 3F: unperturbed), the unperturbed value reaches its group's lanes by shuffle, and every lane turns its F differences
// into matrix contributions.  Every perturbed evaluation is the same operation sequence as in jac_rows_fd (rows_faithful_at
// with the element's own vertex order), so two-term entries keep the oracle's bits.
// No atomics, deterministic: a ring slot receives exactly two contributions -- from the element on either side of the edge
// -- which go to two staging arrays (SA: element k's "this neighbour" column, SB: element k-1's "next neighbour" column)
// and are added at copy-out; diagonal contributions are parked per ring position and summed in ring order.
constexpr int FDW_CHUNK = 64;    // vertices per block pass
constexpr int FDW_CAP = 576;     // staged slots per plane (average valence 8)
constexpr int FDW_KMAX = 16;     // longest ring handled here
constexpr int FDW_WARPS = 8;

// the rare over-long rows: kept out of line so that its register appetite does not shape the kernel's allocation
template <int OP>
__device__ __noinline__ void jacobian_row_fd_slow(const StarView& M, const PhysParams& P, const double* u, const double* aux0,
                                                  const double* aux1, double eps, int comp0, int v, double* vals, long stride) {
  jacobian_row<OP, JAC_FD_FAITHFUL>(M, P, u, aux0, aux1, eps, comp0, v, vals, stride);
}

template <int OP>
__global__ void __launch_bounds__(FDW_WARPS * 32, 2)
k_jacobian_fdw(StarView M, PhysParams P, const double* __restrict__ u, const double* __restrict__ aux0,
               const double* __restrict__ aux1, double eps, int comp0, double* __restrict__ vals, long stride) {
  constexpr int NP = OpTraits<OP>::NPLANES, F = OpTraits<OP>::F, NA = VData<OP>::NA;
  constexpr int NC = 3 * F, TPE = NC + 1, EPR = 32 / TPE; // columns, tasks per element, elements per round
  extern __shared__ double fdw_sm[];
  double* SA = fdw_sm;
  double* SB = fdw_sm + NP * FDW_CAP;
  double* DG = fdw_sm + 2 * NP * FDW_CAP; // [warp][ring position][plane]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane / TPE, c = lane % TPE;
  const int nchunks = (M.nv + FDW_CHUNK - 1) / FDW_CHUNK;
  for (int ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int v0 = ch * FDW_CHUNK, v1 = min(v0 + FDW_CHUNK, M.nv);
    const int sb = M.rp[v0], n = M.rp[v1] - sb;
    int bad = n > FDW_CAP;
    for (int v = v0 + threadIdx.x; v < v1; v += blockDim.x) bad |= (M.rp[v + 1] - M.rp[v] - 1 > FDW_KMAX);
    if (__syncthreads_or(bad)) { // over-long rows: the per-vertex routine writes them directly
      const int v = v0 + threadIdx.x;
      if (v < v1) jacobian_row_fd_slow<OP>(M, P, u, aux0, aux1, eps, comp0, v, vals, stride);
      continue;
    }
    for (int i = threadIdx.x; i < NP * FDW_CAP; i += blockDim.x) { SA[i] = 0.0; SB[i] = 0.0; }
    __syncthreads();
    for (int v = v0 + warp; v < v1; v += FDW_WARPS) {
      const int sd = M.rp[v], s0 = sd + 1, s1 = M.rp[v + 1], nring = s1 - s0;
      const unsigned rb = dir_bits<OP>(M, v, comp0);
      double* dg = DG + warp * FDW_KMAX * NP;
      for (int i = lane; i < FDW_KMAX * NP; i += 32) dg[i] = 0.0;
      __syncwarp();
      if (nring > 0) {
        const VData<OP> V = load_vertex<OP>(M, u, aux0, aux1, v);
        const bool closed = (M.adj[s1 - 1] & STAR_HAS_TRI) != 0;
        for (int k0 = 0; k0 < nring; k0 += EPR) {
          const int k = k0 + g;
          const bool active = g < EPR && k < nring;
          const unsigned a_cur = active ? M.adj[s0 + k] : 0u;
          const bool has = active && (a_cur & STAR_HAS_TRI);
          double res[F], delta = 1.0;
#pragma unroll
          for (int ki = 0; ki < F; ki++) res[ki] = 0.0;
          int li = 0; bool cw = false; unsigned cb_cur = 0, cb_nxt = 0;
          if (has) {
            const bool last = k + 1 == nring;
            const unsigned a_nxt = last ? M.adj[s0] : M.adj[s0 + k + 1];
            const int wc = (int)(a_cur & STAR_VMASK), wn = (int)(a_nxt & STAR_VMASK);
            const VData<OP> cur = load_vertex<OP>(M, u, aux0, aux1, wc), nxt = load_vertex<OP>(M, u, aux0, aux1, wn);
            cb_cur = dir_bits<OP>(M, wc, comp0); cb_nxt = dir_bits<OP>(M, wn, comp0);
            li = (a_cur >> STAR_LI_SHIFT) & 3; cw = (a_cur & STAR_CW) != 0;
            // element-local order: a[li] = v, a[(li+1)%3] = N, a[(li+2)%3] = Pp with (N, Pp) = cw ? (nxt, cur) : (cur, nxt);
            // scalar selects (whole-struct selects end up in local memory)
            const int pN = (li + 1) % 3;
#define pick(pos, fv, fc, fn) ((pos) == li ? (fv) : ((((pos) == pN) != cw) ? (fc) : (fn))) /* position pN holds N: cur unless cw */
            double xl[F][3], aux[NA][3], px[3], py[3];
#pragma unroll
            for (int pos = 0; pos < 3; pos++) {
              px[pos] = pick(pos, V.x, cur.x, nxt.x); py[pos] = pick(pos, V.y, cur.y, nxt.y);
#pragma unroll
              for (int kk = 0; kk < F; kk++) xl[kk][pos] = pick(pos, V.u[kk], cur.u[kk], nxt.u[kk]);
#pragma unroll
              for (int aa = 0; aa < NA; aa++) aux[aa][pos] = pick(pos, V.a[aa], cur.a[aa], nxt.a[aa]);
            }
#undef pick
            const Geo G = make_geo(px[0], py[0], px[1], py[1], px[2], py[2]);
            if (c < NC) { // perturb local dof c = 3*kj + jl (child-major order of NumericalJacobianVolume)
              double keep = 0.0;
#pragma unroll
              for (int kk = 0; kk < F; kk++)
#pragma unroll
                for (int i = 0; i < 3; i++) if (3 * kk + i == c) keep = xl[kk][i];
              delta = eps * (1.0 + fabs(keep));
#pragma unroll
              for (int kk = 0; kk < F; kk++)
#pragma unroll
                for (int i = 0; i < 3; i++) if (3 * kk + i == c) xl[kk][i] = keep + delta;
            }
            rows_faithful_at<OP>(G, P, xl, aux, li, res);
          }
          double dn[F];
#pragma unroll
          for (int ki = 0; ki < F; ki++) dn[ki] = __shfl_sync(0xffffffffu, res[ki], min(g, EPR - 1) * TPE + NC);
          if (has && c < NC) {
            const int kj = c / 3, jl = c % 3;
            const int lc = cw ? (li + 2) % 3 : (li + 1) % 3; // element-local index of this ring neighbour
            const unsigned cb = jl == li ? rb : (jl == lc ? cb_cur : cb_nxt);
#pragma unroll
            for (int ki = 0; ki < F; ki++) {
              const int pl = OP == OP_PNP ? pnp_plane(ki, kj) : 0;
              if (pl < 0) continue;
              double d = (res[ki] - dn[ki]) / delta;
              if (((rb >> ki) & 1u) | ((cb >> kj) & 1u)) d = 0.0; // constrained row or column (the diagonal is set below)
              if (jl == li) dg[k * NP + pl] = d;
              else if (jl == lc) SA[pl * FDW_CAP + (s0 + k - sb)] = d;
              else SB[pl * FDW_CAP + ((k + 1 == nring ? s0 : s0 + k + 1) - sb)] = d;
            }
          }
        }
        (void)closed;
      }
      __syncwarp();
      if (lane < NP) { // diagonal: ring order, as the sequential walk adds it
        double acc = 0.0;
        for (int k = 0; k < nring; k++) acc += dg[k * NP + lane];
        if (OP == OP_PNP) {
          const int ki = lane < 3 ? 0 : (lane < 5 ? 1 : 2), kj = lane < 3 ? lane : (lane == 3 ? 0 : (lane == 4 ? 1 : (lane == 5 ? 0 : 2)));
          if (((rb >> ki) & 1u) | ((rb >> kj) & 1u)) acc = (ki == kj && ((rb >> ki) & 1u)) ? 1.0 : 0.0;
        } else if (rb & 1u) acc = 1.0;
        SA[lane * FDW_CAP + (sd - sb)] = acc;
      }
      __syncwarp();
    }
    __syncthreads();
#pragma unroll
    for (int p = 0; p < NP; p++)
      for (int i = threadIdx.x; i < n; i += blockDim.x) vals[p * stride + sb + i] = SB[p * FDW_CAP + i] + SA[p * FDW_CAP + i];
    __syncthreads();
  }
}

template <int OP>
void launch_jac_fdw(Ctx& c, const StarView& M, const Operator& op, const double* u, const double* a0, const double* a1,
                    double* vals, long stride, double eps) {
  const PhysParams P = c.phys(op.valency);
  constexpr int NP = OpTraits<OP>::NPLANES;
  const int smem = (2 * NP * FDW_CAP + FDW_WARPS * FDW_KMAX * NP) * (int)sizeof(double);
  PNP_CUDA(cudaFuncSetAttribute(k_jacobian_fdw<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int grid = grid_for(M.nv, FDW_CHUNK, c.sm_count * 12);
  k_jacobian_fdw<OP><<<grid, FDW_WARPS * 32, smem, c.stream>>>(M, P, u, a0, a1, eps, op.comp0, vals, stride);
  PNP_CHECK_LAUNCH(); c.launches++;
  c.acct(Ctx::ACC_ASSEMBLY, (4.0 + 8.0 * NP) * (double)stride + (21.0 + 8.0 * OpTraits<OP>::F + 8.0 * OpTraits<OP>::NAUX) * (double)M.nv);
}

} // namespace

#ifdef PNP_ASM_FAITHFUL

void launch_jacobian_fd(Ctx& c, const StarView& M, const Operator& op, const double* u, const double* a0, const double* a1,
                        double* vals, long stride, double eps) {
  if (!tune().fd_warp) { dispatch_jac<JAC_FD_FAITHFUL>(c, M, op, u, a0, a1, vals, stride, eps, op_planes(op.op)); return; }
  switch (op.op) {
    case OP_PB: launch_jac_fdw<OP_PB>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_POISSON: launch_jac_fdw<OP_POISSON>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_DIFFUSION: launch_jac_fdw<OP_DIFFUSION>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_MASS: launch_jac_fdw<OP_MASS>(c, M, op, u, a0, a1, vals, stride, eps); break;
    case OP_PNP: launch_jac_fdw<OP_PNP>(c, M, op, u, a0, a1, vals, stride, eps); break;
    default: PNP_REQUIRE(false, PNP_E_ARG, "unknown operator");
  }
}

#else

namespace {

template <int OP>
__global__ void __launch_bounds__(128)
k_residual(StarView M, PhysParams P, const double* __restrict__ u, const double* __restrict__ aux0,
           const double* __restrict__ aux1, int comp0, double* __restrict__ r) {
  constexpr int F = OpTraits<OP>::F;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < M.nv; v += gridDim.x * blockDim.x) {
    double out[F];
    residual_row<OP, false>(M, P, u, aux0, aux1, v, out);
    const unsigned db = dir_bits<OP>(M, v, comp0);
#pragma unroll
    for (int k = 0; k < F; k++) r[(long)F * v + k] = ((db >> k) & 1u) ? 0.0 : out[k]; // constrain_residual
  }
}

// alpha_boundary: one thread per vertex that occurs in a boundary face (boundary_vertex_sum, pnp_star.cuh)
__global__ void k_boundary(StarView M, PhysParams P, const BFace* __restrict__ faces, const int* __restrict__ bv,
                           const int* __restrict__ ptr, const int* __restrict__ items, int n_bv,
                           const double* __restrict__ surf_flux, const unsigned char* __restrict__ surf_dir, int F,
                           int comp0, double* __restrict__ r) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_bv) return;
  double acc[3];
  boundary_vertex_sum(M, P, faces, items, ptr[t], ptr[t + 1], surf_flux, surf_dir, F, comp0, acc);
  const int v = bv[t];
  const unsigned m = M.dmask[v];
  for (int k = 0; k < F; k++) {
    const int comp = F == 3 ? k : comp0;
    if (!((m >> comp) & 1u)) r[(long)F * v + k] += acc[k];
  }
}

} // namespace
static void coefficient_ptrs(Ctx& c, const Operator& op, const double** a0, const double** a1) {
  *a0 = *a1 = nullptr;
  const int need = op.op == OP_POISSON ? 2 : (op.op == OP_DIFFUSION ? 1 : 0);
  if (need >= 1) {
    PNP_REQUIRE(op.aux0 >= 0, PNP_E_ARG, "operator coefficient 0 not set");
    PNP_REQUIRE(c.vec(op.aux0).fields == 1, PNP_E_ARG, "coefficient must be a 1-field vector");
    *a0 = c.vec(op.aux0).d.p;
  }
  if (need >= 2) {
    PNP_REQUIRE(op.aux1 >= 0, PNP_E_ARG, "operator coefficient 1 not set");
    PNP_REQUIRE(c.vec(op.aux1).fields == 1, PNP_E_ARG, "coefficient must be a 1-field vector");
    *a1 = c.vec(op.aux1).d.p;
  }
  // partitioned mesh: the coefficient fields are read at ghost vertices too, and solver results only cover owned dofs
  if (c.n_own < c.nv) {
    if (*a0) halo_exchange(c, const_cast<double*>(*a0), 1);
    if (*a1) halo_exchange(c, const_cast<double*>(*a1), 1);
  }
}

void assemble_residual(Ctx& c, const Operator& op, Vec& u, Vec& r) {
  PNP_REQUIRE(c.constraints_built, PNP_E_ARG, "constraints not built (mesh finalized + parameters set?)");
  if (c.degree >= 2) { p2_assemble_residual(c, op, u, r); return; }
  const int F = op_fields(op.op);
  PNP_REQUIRE(u.fields == F && r.fields == F, PNP_E_ARG, "vector field count does not match the operator");
  const double *a0, *a1;
  coefficient_ptrs(c, op, &a0, &a1);
  const StarView M = c.star();
  const PhysParams P = c.phys(op.valency);
  const int block = 128, grid = grid_for(c.n_own, block, c.sm_count * 16);
  halo_exchange(c, u.d.p, F); // ghost values of the state (no-op on one GPU)
  switch (op.op) {
    case OP_PB: k_residual<OP_PB><<<grid, block, 0, c.stream>>>(M, P, u.d.p, a0, a1, op.comp0, r.d.p); break;
    case OP_POISSON: k_residual<OP_POISSON><<<grid, block, 0, c.stream>>>(M, P, u.d.p, a0, a1, op.comp0, r.d.p); break;
    case OP_DIFFUSION: k_residual<OP_DIFFUSION><<<grid, block, 0, c.stream>>>(M, P, u.d.p, a0, a1, op.comp0, r.d.p); break;
    case OP_MASS: k_residual<OP_MASS><<<grid, block, 0, c.stream>>>(M, P, u.d.p, a0, a1, op.comp0, r.d.p); break;
    case OP_PNP: k_residual<OP_PNP><<<grid, block, 0, c.stream>>>(M, P, u.d.p, a0, a1, op.comp0, r.d.p); break;
    default: PNP_REQUIRE(false, PNP_E_ARG, "unknown operator");
  }
  PNP_CHECK_LAUNCH(); c.launches++;
  c.acct(Ctx::ACC_ASSEMBLY, 4.0 * (double)c.nslots + (21.0 + 16.0 * F + 8.0 * (op.op == OP_POISSON ? 2 : (op.op == OP_DIFFUSION ? 1 : 0))) * (double)c.n_own);
  // doAlphaBoundary is false for the diffusion and mass operators (diffusion_operator.hh:34)
  if ((op.op == OP_PB || op.op == OP_POISSON || op.op == OP_PNP) && c.n_bv > 0) {
    // Poisson is constructed with the PB BCType (component 0): instationary_pnp_from_pb_md.hh:343-344
    k_boundary<<<(c.n_bv + 127) / 128, 128, 0, c.stream>>>(M, P, c.d_bfaces.p, c.d_bv.p, c.d_bv_ptr.p, c.d_bv_items.p,
                                                          c.n_bv, c.d_surf.p, c.d_surf_dir.p, F, op.comp0, r.d.p);
    PNP_CHECK_LAUNCH(); c.launches++;
  }
}

void assemble_jacobian(Ctx& c, const Operator& op, Vec& u, Matrix& A, int mode, double eps) {
  PNP_REQUIRE(c.constraints_built, PNP_E_ARG, "constraints not built (mesh finalized + parameters set?)");
  if (c.degree >= 2) { p2_assemble_jacobian(c, op, u, A, mode, eps); return; }
  PNP_REQUIRE(u.fields == op_fields(op.op), PNP_E_ARG, "vector field count does not match the operator");
  PNP_REQUIRE(A.op == op.op, PNP_E_ARG, "matrix belongs to another operator type");
  PNP_REQUIRE(mode == JAC_FD_FAITHFUL || mode == JAC_ANALYTIC, PNP_E_ARG, "unknown jacobian mode");
  PNP_REQUIRE(A.nplanes == op_planes(op.op) || (A.nplanes == PNP_COMPACT_PLANES && op.op == OP_PNP && mode == JAC_ANALYTIC),
              PNP_E_ARG, "matrix layout does not fit the operator and Jacobian mode");
  const double *a0, *a1;
  coefficient_ptrs(c, op, &a0, &a1);
  A.comp0 = op.comp0;
  c.last_u = u.d.p; c.last_op = op; c.last_mode = mode; c.last_eps = eps; c.last_vals = A.vals.p;
  halo_exchange(c, u.d.p, u.fields);
  if (mode == JAC_FD_FAITHFUL) launch_jacobian_fd(c, c.star(), op, u.d.p, a0, a1, A.vals.p, c.nslots, eps);
  else dispatch_jac<JAC_ANALYTIC>(c, c.star(), op, u.d.p, a0, a1, A.vals.p, c.nslots, eps, A.nplanes);
}

// The same operator on another star of the same mesh hierarchy (a coarser refinement level held by the multigrid):
// u in that level's numbering, vals = `nplanes` planes of `stride` slots (the layout of the finest level's matrix).
// Operators with coefficient fields are not supported here (their coefficients live on the finest level only).
void assemble_jacobian_on(Ctx& c, const StarView& M, long stride, const Operator& op, const double* u, double* vals, int nplanes,
                          int mode, double eps) {
  PNP_REQUIRE(op.op == OP_PB || op.op == OP_PNP || op.op == OP_MASS, PNP_E_ARG, "no coefficient fields on coarse levels");
  PNP_REQUIRE(nplanes == op_planes(op.op) || (nplanes == PNP_COMPACT_PLANES && op.op == OP_PNP && mode == JAC_ANALYTIC),
              PNP_E_ARG, "matrix layout does not fit the operator and Jacobian mode");
  if (mode == JAC_FD_FAITHFUL) launch_jacobian_fd(c, M, op, u, nullptr, nullptr, vals, stride, eps);
  else dispatch_jac<JAC_ANALYTIC>(c, M, op, u, nullptr, nullptr, vals, stride, eps, nplanes);
}

#endif // PNP_ASM_FAITHFUL

} // namespace pnp
