// pnp_amg.cu -- aggregation AMG preconditioner on the device (PNP_PREC_AMG).
//
// Stands in for Dune::Amg::AMG as selected by ISTLBackend_NOVLP_CG_AMG_SSOR
// (/root/reference/src/instationary_pnp_from_pb_md.hh:208-211; SURVEY.md App. A.8): unsmoothed
// aggregation, Galerkin coarse operators, V-cycle, `prec_steps` smoothing sweeps before and after the
// coarse correction, coarse correction scaled by dune-istl's default prolongation damping 1.6.
// What differs, because the sequential pieces of ISTL have no parallel equivalent: aggregates come
// from a parallel maximal independent set (root + its strongest-coupled neighbours) instead of
// ISTL's sequential front-growing, and the smoother is damped Jacobi instead of SSOR.  Linear
// iteration counts therefore differ from ISTL's; Newton counts do not (SURVEY H3).
//
// Point-block hierarchy: all fields of a vertex are aggregated together, so every level keeps the
// 1-plane (scalar), 7-plane or compact 5-plane (PNP) layout of the fine matrix and runs the same SpMV.  The Galerkin sums
// are linear in the planes, so a compact level's coarse operator is the compact form of the 7-plane one.
// Symbolic phase (aggregates, coarse patterns, gather lists) once per mesh/operator type;
// numeric phase (Galerkin sums, inverse diagonals) per Jacobian -- deterministic gathers, no atomics.
#include <cub/cub.cuh>
#include <cusolverDn.h>

#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "pnp_common.cuh"
#include "pnp_spmv_tma.cuh"
#include "pnp_sweep.cuh"

namespace pnp {

// pnp_precond.cu: level schedule of a row-order sweep on a star-layout matrix, one Gauss-Seidel sweep along / against it
std::shared_ptr<SweepPlan> sweep_plan_build(Ctx&, const SweepView&, int F);
void sweep_gs(Ctx&, const SweepPlan&, const SweepView&, const double* vals, long stride, const double* d, double* x, int dir);

namespace {

constexpr int BLK = 256;

struct Level {
  int nv = 0; long nslots = 0;
  // matrix (level 0 borrows the context's star arrays and the caller's values)
  const int* rp = nullptr; const unsigned* col = nullptr; const double* vals = nullptr;
  DBuf<int> rp_own; DBuf<unsigned> col_own; DBuf<double> vals_own;
  DBuf<double> dinv, x, x2, b, r;
  // single-precision companion of `vals` (empty: none, mg_f32_rule()): the same planes rounded to nearest, stride32 (a
  // multiple of 4) floats apart so that every plane starts on a 16-byte boundary.  Where it exists, every operation of
  // the smoothing cycle on this level -- the first Jacobi sweep's stored block inverses, the smoother steps and the
  // residual -- applies the rounded matrix (widened to double); the Krylov operator, the Galerkin products, the dense
  // coarsest level and the exports keep reading `vals`.  Rebuilt from `vals` by every numeric set-up, never written
  // anywhere else, so it cannot go stale when the caller's planes change.
  DBuf<float> vals32; long stride32 = 0;
  double lmax = 2.0;      // Gershgorin bound of the spectrum of D^-1 A
  // transfer to the next coarser level
  // Prolongation row of fine vertex i: one parent (weight 1: aggregate / coinciding coarse vertex) or two parents
  // (weight 1/2 each: midpoint of a coarse edge, P1 interpolation of the refinement hierarchy).
  DBuf<int> agg, par1;               // first parent; second parent or -1 (par1 empty: aggregation level)
  DBuf<int> agg_ptr, agg_mem;        // coarse vertex -> fine vertices it is a parent of (restriction = P^T)
  DBuf<int> seg_ptr, seg_items;      // coarse slot -> fine slots summed into it (Galerkin P^T A P)
  DBuf<unsigned char> seg_w;         // weight code of each item: 0 -> 1, 1 -> 1/2, 2 -> 1/4 (empty: all 1)
  double alpha = 1.0;                // scaling of the coarse correction coming up from the next level
  // distributed geometric level: the context that owns this level's mesh part (halo plan, Dirichlet mask); coarse
  // levels are re-discretised on it from the injected state u
  Ctx* lc = nullptr;
  Vec u; Matrix Amat;
  // Dirichlet mask of the level's OWN vertices: level 0, distributed levels and re-discretised geometric levels keep
  // their constrained dofs (identity rows); null for Galerkin / aggregation levels, which carry none of their own
  const unsigned char* dm = nullptr;
  // geometric level of a one-GPU hierarchy whose operator is re-discretised on its own star (coordinates and mask
  // gathered from the finest level, state u injected) instead of the Galerkin product
  bool redisc = false;
  DBuf<XY> xy_own; DBuf<unsigned char> dmask_own;
  std::shared_ptr<SweepPlan> gs_plan; // Gauss-Seidel smoother: level schedule of this level's rows (built on first use)
};

} // namespace

struct Amg {
  int NP = 1, F = 1;
  bool symbolic = false;
  long nv0 = -1, nslots0 = -1;
  long mg_epoch = -1;       // Ctx::mg_epoch the hierarchy was built for
  double sym_key = 0.0;     // the options that shape the hierarchy (a change rebuilds it)
  double omega = 0.7, alpha = 1.6;
  int coarse_sweeps = 40;
  int gamma = 1;          // 1: V-cycle, 2: W-cycle ...
  int wlevels = 99;       // ... on the first `wlevels` levels only (V below): bounds the visits of the small levels
  int smoother = 0;       // 0: damped Jacobi, 1: Chebyshev on [lmax/cheb_ratio, lmax] of D^-1 A, 2: symmetric Gauss-Seidel (SSOR, w = 1)
  double cheb_ratio = 8.0;
  int comp0 = 0;
  int pre_steps = -1, post_steps = -1; // smoothing steps before / after the coarse correction (-1: the solver's prec_steps)
  // coarsest level: dense LU (cuSOLVER getrf/getrs) when it has at most dense_max dofs, else `coarse_sweeps` sweeps
  int dense_max = 4096, dense_n = 0;
  cusolverDnHandle_t cus = nullptr;
  DBuf<double> dense, dense_work;
  DBuf<int> dense_piv, dense_info;
  bool distributed = false; // levels are parts of a mesh hierarchy spread over the ranks (halo exchange per level)
  bool replica = false;     // the single-GPU hierarchy below a distributed one's replicated coarsest level (rep_solver)
  bool redisc = false;      // one GPU: the geometric levels are re-discretised (as the distributed levels are), not Galerkin products
  DBuf<double> grhs;        // replicated coarsest level: global right-hand side / solution
  // replica variant (Ctx::mg_replica): the coarsest distributed level is gathered to a context that holds the whole
  // coarsest mesh; that context runs its own (single-GPU) hierarchy below: aggregation levels + small dense LU
  std::unique_ptr<Solver> rep_solver; Matrix rep_A; Vec rep_u; DBuf<double> rep_x;
  int n_geo = 0;          // number of geometric (P1) transfers at the top of the hierarchy
  std::vector<std::unique_ptr<Level>> L;
  DBuf<unsigned char> tmp;
  void* temp(size_t bytes) { if (bytes > tmp.n) tmp.alloc(bytes); return tmp.p; }
  // CUDA graph of the coarse correction (everything below the finest level of one cycle: ~80 small launches that are
  // launch-latency bound, the more so the more GPUs share the mesh).  Captured at the second application, replayed after;
  // the iterate pointers the smoothers swap are put back to their state at capture before every replay.
  cudaGraphExec_t cg_exec = nullptr;
  bool cg_failed = false;
  int cg_calls = 0;
  double cg_key[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::vector<std::pair<double*, double*>> cg_before, cg_after;
  long cg_launches = 0; double cg_bytes[Ctx::ACC_N] = {0, 0, 0, 0, 0, 0};
  void cg_reset() { if (cg_exec) cudaGraphExecDestroy(cg_exec); cg_exec = nullptr; cg_calls = 0; }
  ~Amg() { if (cg_exec) cudaGraphExecDestroy(cg_exec); if (cus) cusolverDnDestroy(cus); }
};

namespace {

__device__ __forceinline__ unsigned hash32(unsigned x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
// Luby rounds. state: 0 undecided, 1 root, 2 covered
__global__ void k_mis_select(const int* __restrict__ rp, const unsigned* __restrict__ col, int nv,
                             const unsigned char* __restrict__ st, unsigned char* __restrict__ st_out) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    unsigned char s = st[v];
    if (s == 0) {
      const unsigned pv = hash32((unsigned)v);
      bool win = true;
      for (int k = rp[v] + 1; k < rp[v + 1]; k++) {
        const int w = (int)(col[k] & STAR_VMASK);
        if (w >= nv || w == v || st[w] != 0) continue; // (ghost columns take no part in the local hierarchy)
        const unsigned pw = hash32((unsigned)w);
        if (pw > pv || (pw == pv && w > v)) { win = false; break; }
      }
      if (win) s = 1;
    }
    st_out[v] = s;
  }
}
__global__ void k_mis_cover(const int* __restrict__ rp, const unsigned* __restrict__ col, int nv,
                            unsigned char* __restrict__ st, int* __restrict__ undecided) {
  int local = 0;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    if (st[v] != 0) continue;
    bool covered = false;
    for (int k = rp[v] + 1; k < rp[v + 1]; k++) {
      const int w = (int)(col[k] & STAR_VMASK);
      if (w < nv && st[w] == 1) { covered = true; break; }
    }
    if (covered) st[v] = 2; else local++;
  }
  if (local) atomicAdd(undecided, local);
}
__global__ void k_root_flag(const unsigned char* __restrict__ st, int nv, int* __restrict__ flag) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) flag[v] = st[v] == 1;
}
// every covered vertex joins the adjacent root it is most strongly coupled to (|plane 0|)
__global__ void k_attach(const int* __restrict__ rp, const unsigned* __restrict__ col, const double* __restrict__ vals,
                         int nv, const unsigned char* __restrict__ st, const int* __restrict__ root_id,
                         int* __restrict__ agg) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    if (st[v] == 1) { agg[v] = root_id[v]; continue; }
    double best = -1.0; int bw = -1;
    for (int k = rp[v] + 1; k < rp[v + 1]; k++) {
      const int w = (int)(col[k] & STAR_VMASK);
      if (w >= nv || st[w] != 1) continue;
      const double s = fabs(vals[k]);
      if (s > best || (s == best && w < bw)) { best = s; bw = w; }
    }
    agg[v] = root_id[bw];
  }
}
// coarse-slot key of every fine slot: (I << 32) | (J == I ? 0 : J + 1)  -> the diagonal sorts first
__global__ void k_coarse_keys(const int* __restrict__ rp, const unsigned* __restrict__ col, int nv,
                              const int* __restrict__ agg, uint64_t* __restrict__ keys, int* __restrict__ slot_id) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    const unsigned I = (unsigned)agg[v];
    for (int k = rp[v]; k < rp[v + 1]; k++) {
      const unsigned w = col[k] & STAR_VMASK;
      if (w >= (unsigned)nv) { keys[k] = ~0ull; slot_id[k] = k; continue; } // ghost column: dropped (block-Jacobi over ranks)
      const unsigned J = (unsigned)agg[w];
      keys[k] = ((uint64_t)I << 32) | (J == I ? 0u : J + 1u);
      slot_id[k] = k;
    }
  }
}
__global__ void k_coarse_cols(const uint64_t* __restrict__ ukeys, long n, unsigned* __restrict__ col) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const unsigned lo = (unsigned)(ukeys[i] & 0xffffffffu);
    col[i] = lo == 0 ? (unsigned)(ukeys[i] >> 32) : lo - 1u;
  }
}
__global__ void k_row_starts(const uint64_t* __restrict__ ukeys, long n, int nc, int* __restrict__ rp) {
  for (int I = blockIdx.x * blockDim.x + threadIdx.x; I <= nc; I += gridDim.x * blockDim.x)
    rp[I] = (int)lower_bound_u64(ukeys, n, (uint64_t)(unsigned)I << 32);
}
__global__ void k_lower_bounds_i32(const int* __restrict__ sorted, int n, int m, int* __restrict__ out) {
  for (int I = blockIdx.x * blockDim.x + threadIdx.x; I <= m; I += gridDim.x * blockDim.x) {
    int lo = 0, hi = n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (sorted[mid] < I) lo = mid + 1; else hi = mid; }
    out[I] = lo;
  }
}
__global__ void k_iota(int* a, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) a[i] = i;
}

// Galerkin sums A_c = P^T A P for piecewise-constant P: coarse slot cs = sum of its fine slots.
// At level 0 Dirichlet dofs are left out of the hierarchy (their rows/columns are already decoupled;
// only the unit diagonal has to be skipped): dmask/rp0 non-null, F = 3 uses bits 0..2, F = 1 uses bit comp0.
template <int NP>
__global__ void k_galerkin(const int* __restrict__ seg_ptr, const int* __restrict__ seg_items,
                           const unsigned char* __restrict__ seg_w, long nsc, const double* __restrict__ vf, long nsf, double* __restrict__ vc,
                           const unsigned char* __restrict__ dmask, const unsigned* __restrict__ colf, const int* __restrict__ rpf,
                           int comp0) {
  for (long cs = blockIdx.x * (long)blockDim.x + threadIdx.x; cs < nsc; cs += (long)gridDim.x * blockDim.x) {
    double acc[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) acc[p] = 0.0;
    // items are taken four at a time: the four slot indices first, then all 4*NP value loads, so that the scattered
    // gathers of one thread overlap (a coarse slot of a refinement level has ~12 items; one at a time the loop is a
    // chain of dependent index -> value round trips).  The summation order is the item order, as before.
    constexpr int U = 4;
    const int t1 = seg_ptr[cs + 1];
    for (int t0 = seg_ptr[cs]; t0 < t1; t0 += U) {
      int s[U]; double w[U]; double v[U][NP];
#pragma unroll
      for (int q = 0; q < U; q++) {
        const bool ok = t0 + q < t1;
        s[q] = ok ? seg_items[t0 + q] : -1;
        const unsigned char wc = (ok && seg_w) ? seg_w[t0 + q] : 0;
        w[q] = ok ? (wc == 0 ? 1.0 : (wc == 1 ? 0.5 : 0.25)) : 0.0;
      }
#pragma unroll
      for (int q = 0; q < U; q++)
#pragma unroll
        for (int p = 0; p < NP; p++) v[q][p] = s[q] >= 0 ? vf[p * nsf + s[q]] : 0.0;
      if (dmask) { // level 0: skip the unit diagonal of constrained dofs (slot s is a diagonal slot iff s == rp[col[s]])
#pragma unroll
        for (int q = 0; q < U; q++) {
          if (s[q] < 0) continue;
          const unsigned wv = colf[s[q]] & STAR_VMASK;
          const unsigned m = dmask[wv];
          if (m && rpf[wv] == s[q]) {
            if (NP == 1) { if ((m >> comp0) & 1u) v[q][0] = 0.0; }
            else if (NP == PNP_COMPACT_PLANES) { if (m & 1u) v[q][0] = 0.0; } // all three fields: L = 1, D = 0
            else {
              if (m & 1u) v[q][0] = 0.0;
              if (m & 2u) v[q][NP == 7 ? 4 : 0] = 0.0;
              if (m & 4u) v[q][NP == 7 ? 6 : 0] = 0.0;
            }
          }
        }
      }
#pragma unroll
      for (int q = 0; q < U; q++)
        if (s[q] >= 0) {
#pragma unroll
          for (int p = 0; p < NP; p++) acc[p] += w[q] * v[q][p];
        }
    }
#pragma unroll
    for (int p = 0; p < NP; p++) vc[p * nsc + cs] = acc[p];
  }
}
// smoother matrix M^-1: scalar operators 1/a_ii; PNP: inverse of every vertex's 3x3 diagonal block (point-block Jacobi --
// the phi/c couplings inside a vertex grow like h^2 relative to the stiffness terms, so on coarse levels a scalar
// diagonal no longer dominates them)
template <int NP, class T>
__global__ void k_dinv(const int* __restrict__ rp, const T* __restrict__ vals, long stride, int nv,
                       double* __restrict__ dinv) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    const int s = rp[v];
    if (NP == 1) { const double d = vals[s]; dinv[v] = d != 0.0 ? 1.0 / d : 0.0; }
    else {
      // B = [a b c; d e 0; f 0 g] (float planes widened first: the block of the rounded matrix, inverted in double)
      double pv[NP];
#pragma unroll
      for (int p = 0; p < NP; p++) pv[p] = vals[p * stride + s];
      const PnpBlock B = pnp_block<NP>(pv);
      const double a = B.a, b = B.b, c_ = B.c, d = B.d, e = B.e, f = B.f, g = B.g;
      const double det = a * e * g - b * d * g - c_ * e * f;
      double* o = dinv + 9l * v;
      const double scale = fabs(a * e * g) + fabs(b * d * g) + fabs(c_ * e * f);
      if (fabs(det) > 1e-12 * scale && scale > 0.0) {
        const double id = 1.0 / det;
        o[0] = e * g * id;   o[1] = -b * g * id;           o[2] = -c_ * e * id;
        o[3] = -d * g * id;  o[4] = (a * g - c_ * f) * id; o[5] = c_ * d * id;
        o[6] = -e * f * id;  o[7] = b * f * id;            o[8] = (a * e - b * d) * id;
      } else { // (near-)singular block, e.g. an all-Dirichlet coarse vertex: fall back to the scalar diagonal
        for (int i = 0; i < 9; i++) o[i] = 0.0;
        o[0] = a != 0.0 ? 1.0 / a : 0.0; o[4] = e != 0.0 ? 1.0 / e : 0.0; o[8] = g != 0.0 ? 1.0 / g : 0.0;
      }
    }
  }
}
// single-precision companion of a level's planes: o[p * stride32 + s] = fl32(v[p * stride + s]), zero in the padding
__global__ void k_round_planes(const double* __restrict__ v, long stride, long ns, float* __restrict__ o, long stride32) {
  const double* vp = v + blockIdx.y * stride;
  float* op = o + blockIdx.y * stride32;
  for (long s = blockIdx.x * (long)blockDim.x + threadIdx.x; s < stride32; s += (long)gridDim.x * blockDim.x)
    op[s] = s < ns ? __double2float_rn(vp[s]) : 0.0f;
}
// first sweep from a zero initial guess: x = omega * M^-1 b  (also the first Chebyshev direction d)
template <int F>
__global__ void k_jacobi0(const double* __restrict__ dinv, const double* __restrict__ b, double omega,
                          double* __restrict__ x, int nv, double* __restrict__ dvec) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    if (F == 1) {
      const double z = omega * dinv[v] * b[v];
      x[v] = z; if (dvec) dvec[v] = z;
    } else {
      const double* B = dinv + 9l * v;
      const double r0 = b[3l * v], r1 = b[3l * v + 1], r2 = b[3l * v + 2];
#pragma unroll
      for (int k = 0; k < 3; k++) {
        const double z = omega * (B[3 * k] * r0 + B[3 * k + 1] * r1 + B[3 * k + 2] * r2);
        x[3l * v + k] = z; if (dvec) dvec[3l * v + k] = z;
      }
    }
  }
}
// Gershgorin bound of D^-1 A: max over dof rows of sum_j |a_ij| / |a_ii|
template <int NP>
__global__ void k_gershgorin(const int* __restrict__ rp, const double* __restrict__ vals, long stride, int nv,
                             unsigned long long* __restrict__ out) {
  double best = 0.0;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    const int s0 = rp[v], s1 = rp[v + 1];
    if (NP == 1) {
      double sum = 0.0;
      for (int s = s0; s < s1; s++) sum += fabs(vals[s]);
      const double d = fabs(vals[s0]);
      if (d > 0.0) best = fmax(best, sum / d);
    } else {
      double s0_ = 0.0, s1_ = 0.0, s2_ = 0.0;
      for (int s = s0; s < s1; s++) {
        const PnpBlock B = pnp_block_at<NP>(vals, stride, s);
        s0_ += fabs(B.a) + fabs(B.b) + fabs(B.c);
        s1_ += fabs(B.d) + fabs(B.e);
        s2_ += fabs(B.f) + fabs(B.g);
      }
      const PnpBlock D = pnp_block_at<NP>(vals, stride, s0);
      const double d0 = fabs(D.a), d1 = fabs(D.e), d2 = fabs(D.g);
      if (d0 > 0.0) best = fmax(best, s0_ / d0);
      if (d1 > 0.0) best = fmax(best, s1_ / d1);
      if (d2 > 0.0) best = fmax(best, s2_ / d2);
    }
  }
  for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(best)); // positive doubles order like integers
}
template <int F>
__global__ void k_restrict(const int* __restrict__ agg_ptr, const int* __restrict__ agg_mem, const int* __restrict__ par1,
                           int nc, const double* __restrict__ r, double* __restrict__ bc) {
  for (int I = blockIdx.x * blockDim.x + threadIdx.x; I < nc; I += gridDim.x * blockDim.x) {
    double acc[F];
#pragma unroll
    for (int k = 0; k < F; k++) acc[k] = 0.0;
    for (int t = agg_ptr[I]; t < agg_ptr[I + 1]; t++) {
      const long v = agg_mem[t];
      const double w = (par1 && par1[v] >= 0) ? 0.5 : 1.0;
#pragma unroll
      for (int k = 0; k < F; k++) acc[k] += w * r[F * v + k];
    }
#pragma unroll
    for (int k = 0; k < F; k++) bc[(long)F * I + k] = acc[k];
  }
}
// x += alpha * P x_c ; constrained dofs (level 0 only) receive no correction
template <int F>
__global__ void k_prolong(const int* __restrict__ agg, const int* __restrict__ par1, int nv, const double* __restrict__ xc,
                          double alpha, double* __restrict__ x, const unsigned char* __restrict__ dmask, int comp0) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    const long I = agg[v];
    const long J = par1 ? par1[v] : -1;
    const unsigned m = dmask ? (F == 3 ? dmask[v] : (dmask[v] >> comp0) & 1u) : 0u;
#pragma unroll
    for (int k = 0; k < F; k++)
      if (!((m >> k) & 1u))
        x[(long)F * v + k] += alpha * (J >= 0 ? 0.5 * (xc[F * I + k] + xc[F * J + k]) : xc[F * I + k]);
  }
}
// coordinates and Dirichlet mask of a coarser refinement level: a coarse vertex IS a finest-level vertex (same reference index)
__global__ void k_level_geometry(const int* __restrict__ int2ext_c, const int* __restrict__ ext2int_f, const XY* __restrict__ xy_f,
                                 const unsigned char* __restrict__ dmask_f, int nvc, XY* __restrict__ xy_c,
                                 unsigned char* __restrict__ dmask_c) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nvc; i += gridDim.x * blockDim.x) {
    const int j = ext2int_f[int2ext_c[i]];
    xy_c[i] = xy_f[j]; dmask_c[i] = dmask_f[j];
  }
}
// ---- geometric levels: P1 interpolation between two consecutive refinement levels ----
// parents of every fine vertex, both in the internal numbering of their level
__global__ void k_geo_parents(const int* __restrict__ int2ext_f, int nvf, int nvc, const uint64_t* __restrict__ edges,
                              const int* __restrict__ ext2int_c, int* __restrict__ par0, int* __restrict__ par1) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nvf; i += gridDim.x * blockDim.x) {
    const int e = int2ext_f[i];
    if (e < nvc) { par0[i] = ext2int_c[e]; par1[i] = -1; }
    else {
      const uint64_t k = edges[e - nvc];
      par0[i] = ext2int_c[(int)(k >> 32)]; par1[i] = ext2int_c[(int)(k & 0xffffffffu)];
    }
  }
}
// (parent, child) pairs for the restriction lists: 2 per fine vertex, unused ones get key INT_MAX
__global__ void k_geo_pairs(const int* __restrict__ par0, const int* __restrict__ par1, int nvf, int nrows_c,
                            int* __restrict__ key, int* __restrict__ val) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nvf; i += gridDim.x * blockDim.x) {
    key[2 * i] = (par0[i] >= 0 && par0[i] < nrows_c) ? par0[i] : 0x7fffffff; val[2 * i] = i;     // rows of owned coarse vertices only
    key[2 * i + 1] = (par1[i] >= 0 && par1[i] < nrows_c) ? par1[i] : 0x7fffffff; val[2 * i + 1] = i;
  }
}
// injection of the state: a coarse vertex takes the value of the fine vertex it coincides with
template <int F>
__global__ void k_inject(const int* __restrict__ par0, const int* __restrict__ par1, int nvf, const double* __restrict__ uf,
                         double* __restrict__ uc) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nvf; i += gridDim.x * blockDim.x)
    if (par1[i] < 0 && par0[i] >= 0) {
#pragma unroll
      for (int k = 0; k < F; k++) uc[(long)F * par0[i] + k] = uf[(long)F * i + k];
    }
}
template <int F>
__global__ void k_mask_dirichlet(double* __restrict__ b, const unsigned char* __restrict__ dmask, int nv, int comp0) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    const unsigned m = F == 3 ? dmask[v] : (dmask[v] >> comp0) & 1u;
#pragma unroll
    for (int k = 0; k < F; k++) if ((m >> k) & 1u) b[(long)F * v + k] = 0.0;
  }
}
// replicated coarsest level: dense matrix / vectors in GLOBAL dof numbering
template <int NP>
__global__ void k_dense_fill_global(const int* __restrict__ rp, const unsigned* __restrict__ col, const double* __restrict__ vals,
                                    long stride, int nrows, const int* __restrict__ gid, double* __restrict__ Ad, long n,
                                    const unsigned char* __restrict__ dmask, int comp0) {
  constexpr int F = NP == 1 ? 1 : 3;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += gridDim.x * blockDim.x) {
    const long rg = gid[r];
    for (int s = rp[r]; s < rp[r + 1]; s++) {
      const long cg = gid[col[s] & STAR_VMASK];
      // (aggregated coarse system: several entries land on one dense entry; unit diagonals of constrained dofs stay out)
      const unsigned dm = (dmask && s == rp[r]) ? dmask[r] : 0u;
      if (NP == 1) { if (!((dm >> comp0) & 1u)) atomicAdd(&Ad[cg * n + rg], vals[s]); }
      else {
        const PnpBlock B = pnp_block_at<NP>(vals, stride, s);
#pragma unroll
        for (int ki = 0; ki < 3; ki++)
#pragma unroll
          for (int kj = 0; kj < 3; kj++)
            if (pnp_plane(ki, kj) >= 0 && !(ki == kj && ((dm >> ki) & 1u))) atomicAdd(&Ad[(F * cg + kj) * n + F * rg + ki], B.at(ki, kj));
      }
    }
  }
}
template <int F>
__global__ void k_to_global(const double* __restrict__ loc, const int* __restrict__ gid, int nrows, double* __restrict__ glob) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nrows; v += gridDim.x * blockDim.x)
#pragma unroll
    for (int k = 0; k < F; k++) atomicAdd(&glob[(long)F * gid[v] + k], loc[(long)F * v + k]);
}
// x += alpha * (aggregate value), constrained dofs excepted
template <int F>
__global__ void k_add_from_global(const double* __restrict__ glob, const int* __restrict__ gid, int nrows, double alpha,
                                  double* __restrict__ x, const unsigned char* __restrict__ dmask, int comp0) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nrows; v += gridDim.x * blockDim.x) {
    const unsigned m = F == 3 ? dmask[v] : (dmask[v] >> comp0) & 1u;
#pragma unroll
    for (int k = 0; k < F; k++) if (!((m >> k) & 1u)) x[(long)F * v + k] += alpha * glob[(long)F * gid[v] + k];
  }
}
template <int F>
__global__ void k_from_global(const double* __restrict__ glob, const int* __restrict__ gid, int nloc, double* __restrict__ loc) {
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nloc; v += gridDim.x * blockDim.x)
#pragma unroll
    for (int k = 0; k < F; k++) loc[(long)F * v + k] = glob[(long)F * gid[v] + k];
}
__device__ __forceinline__ int find_slot(const int* rp, const unsigned* col, int I, int J) {
  for (int s = rp[I]; s < rp[I + 1]; s++) if ((int)(col[s] & STAR_VMASK) == J) return s;
  return -1;
}
// Galerkin items: fine slot (i,j) feeds coarse slot (I,J) for every parent I of i and J of j with weight w_I*w_J.
// 4 candidate items per fine slot at [4s, 4s+4): key = coarse slot (INT_MAX if unused), val = s | weight code << 29
__global__ void k_geo_items(const int* __restrict__ rpf, const unsigned* __restrict__ colf, int nvf,
                            const int* __restrict__ par0, const int* __restrict__ par1, const int* __restrict__ rpc,
                            const unsigned* __restrict__ colc, int* __restrict__ key, unsigned* __restrict__ val,
                            int* __restrict__ err) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nvf; i += gridDim.x * blockDim.x) {
    const int I[2] = {par0[i], par1[i]};
    for (int s = rpf[i]; s < rpf[i + 1]; s++) {
      const int j = (int)(colf[s] & STAR_VMASK);
      const int J[2] = {par0[j], par1[j]};
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          const long o = 4l * s + 2 * a + b;
          if (I[a] < 0 || J[b] < 0) { key[o] = 0x7fffffff; val[o] = 0; continue; }
          const int cs = find_slot(rpc, colc, I[a], J[b]);
          if (cs < 0) { atomicExch(err, 1); key[o] = 0x7fffffff; val[o] = 0; continue; }
          const unsigned wc = (I[1] >= 0 ? 1u : 0u) + (J[1] >= 0 ? 1u : 0u);
          key[o] = cs; val[o] = (unsigned)s | (wc << 29);
        }
    }
  }
}
__global__ void k_geo_unpack(const unsigned* __restrict__ val, long n, int* __restrict__ items, unsigned char* __restrict__ w) {
  for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < n; t += (long)gridDim.x * blockDim.x) {
    items[t] = (int)(val[t] & 0x1fffffffu); w[t] = (unsigned char)(val[t] >> 29);
  }
}

#define KL(c, kern, n, ...)                                                                              \
  do { kern<<<grid_for((n), BLK), BLK, 0, (c).stream>>>(__VA_ARGS__); PNP_CHECK_LAUNCH(); (c).launches++; } while (0)

template <int EPI>
void level_op(Ctx& c, const Amg& A, const Level& l, const double* x, const double* b, double* y, double omega_or_c2 = -1.0,
              double c1 = 0.0, double* dvec = nullptr) {
  StarOpArgs a{l.rp, l.col, l.vals, l.nslots, l.nv, x, y};
  a.b = b; a.dinv = l.dinv.p; a.block = A.F == 3; a.omega = omega_or_c2 < 0 ? A.omega : omega_or_c2; a.c1 = c1; a.dvec = dvec;
  a.vals32 = l.vals32.p; a.stride32 = l.stride32; // (the one place that picks the planes a cycle operation reads)
  const bool fine = &l == A.L[0].get();
  if (A.distributed) halo_exchange(*l.lc, const_cast<double*>(x), A.F); // ghost columns of the iterate
  if (fine) c.prof_mark(EPI == EPI_RESIDUAL ? 1 : 2);
  launch_star_op_auto<EPI, 0>(c, A.NP, a, fine);
  if (fine) c.prof_mark();
}

// builds level li+1 from level li (symbolic); returns false if coarsening stalled
bool coarsen(Ctx& c, Amg& A, int li) {
  Level& f = *A.L[li];
  const int nv = f.nv;
  DBuf<unsigned char> st(nv), st2(nv);
  st.zero(c.stream);
  DBuf<int> d_und(1);
  for (int round = 0; round < 200; round++) {
    KL(c, k_mis_select, nv, f.rp, f.col, nv, st.p, st2.p);
    std::swap(st.p, st2.p);
    d_und.zero(c.stream);
    KL(c, k_mis_cover, nv, f.rp, f.col, nv, st.p, d_und.p);
    int und = 0;
    d_und.download(&und, 1, c.stream);
    if (und == 0) break;
    PNP_REQUIRE(round < 199, PNP_E_ARG, "AMG: independent-set selection did not terminate");
  }
  DBuf<int> flag(nv), root_id(nv);
  KL(c, k_root_flag, nv, st.p, nv, flag.p);
  size_t bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, flag.p, root_id.p, nv, c.stream);
  PNP_CUDA(cub::DeviceScan::ExclusiveSum(A.temp(bytes), bytes, flag.p, root_id.p, nv, c.stream));
  int last_id = 0, last_flag = 0;
  PNP_CUDA(cudaMemcpyAsync(&last_id, root_id.p + nv - 1, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  PNP_CUDA(cudaMemcpyAsync(&last_flag, flag.p + nv - 1, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  const int nc = last_id + last_flag;
  if (nc < 1 || nc > 0.8 * nv) return false;
  f.alpha = A.alpha;
  f.agg.alloc(nv);
  KL(c, k_attach, nv, f.rp, f.col, f.vals, nv, st.p, root_id.p, f.agg.p);
  // members of each aggregate
  {
    DBuf<int> ids(nv), agg_sorted(nv);
    f.agg_mem.alloc(nv); f.agg_ptr.alloc(nc + 1);
    KL(c, k_iota, nv, ids.p, nv);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, f.agg.p, agg_sorted.p, ids.p, f.agg_mem.p, nv, 0, 32, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortPairs(A.temp(bytes), bytes, f.agg.p, agg_sorted.p, ids.p, f.agg_mem.p, nv, 0, 32,
                                            c.stream));
    KL(c, k_lower_bounds_i32, nc + 1, agg_sorted.p, nv, nc, f.agg_ptr.p);
  }
  // coarse pattern + gather lists
  auto nl = std::make_unique<Level>();
  {
    const long ns = f.nslots;
    PNP_REQUIRE(ns < (1l << 31), PNP_E_MESH, "AMG: too many matrix slots on one level");
    DBuf<uint64_t> keys(ns), skeys(ns), ukeys(ns);
    DBuf<int> slot(ns), counts(ns + 1), d_nu(1);
    f.seg_items.alloc(ns);
    KL(c, k_coarse_keys, nv, f.rp, f.col, nv, f.agg.p, keys.p, slot.p);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys.p, skeys.p, slot.p, f.seg_items.p, (int)ns, 0, 64, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortPairs(A.temp(bytes), bytes, keys.p, skeys.p, slot.p, f.seg_items.p, (int)ns, 0, 64,
                                            c.stream));
    cub::DeviceRunLengthEncode::Encode(nullptr, bytes, skeys.p, ukeys.p, counts.p, d_nu.p, (int)ns, c.stream);
    PNP_CUDA(cub::DeviceRunLengthEncode::Encode(A.temp(bytes), bytes, skeys.p, ukeys.p, counts.p, d_nu.p, (int)ns, c.stream));
    int nu = 0;
    d_nu.download(&nu, 1, c.stream);
    { // the run of dropped ghost-column slots (key ~0) sorts last: leave it out
      uint64_t lastkey = 0;
      PNP_CUDA(cudaMemcpyAsync(&lastkey, ukeys.p + (nu - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost, c.stream));
      PNP_CUDA(cudaStreamSynchronize(c.stream));
      if (lastkey == ~0ull) nu--;
    }
    nl->nv = nc; nl->nslots = nu;
    PNP_CUDA(cudaMemsetAsync(counts.p + nu, 0, sizeof(int), c.stream));
    f.seg_ptr.alloc((size_t)nu + 1);
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, counts.p, f.seg_ptr.p, nu + 1, c.stream);
    PNP_CUDA(cub::DeviceScan::ExclusiveSum(A.temp(bytes), bytes, counts.p, f.seg_ptr.p, nu + 1, c.stream));
    nl->rp_own.alloc((size_t)nc + 1); nl->col_own.alloc(nu);
    KL(c, k_row_starts, nc + 1, ukeys.p, (long)nu, nc, nl->rp_own.p);
    KL(c, k_coarse_cols, nu, ukeys.p, (long)nu, nl->col_own.p);
    c.launches += 8;
    PNP_CUDA(cudaStreamSynchronize(c.stream));
  }
  nl->vals_own.alloc((size_t)A.NP * nl->nslots);
  nl->rp = nl->rp_own.p; nl->col = nl->col_own.p; nl->vals = nl->vals_own.p;
  A.L.push_back(std::move(nl));
  return true;
}

// builds level li+1 from the refinement hierarchy: coarse star = that mesh level's star, P = P1 interpolation
void coarsen_geometric(Ctx& c, Amg& A, int li, const HierLevel& h, const int* int2ext_f, bool redisc) {
  Level& f = *A.L[li];
  const int nvf = f.nv, nvc = (int)h.nv;
  size_t bytes = 0;
  f.agg.alloc(nvf); f.par1.alloc(nvf);
  KL(c, k_geo_parents, nvf, int2ext_f, nvf, nvc, h.edges.p, h.ext2int.p, f.agg.p, f.par1.p);
  { // restriction lists
    DBuf<int> key(2 * (size_t)nvf), val(2 * (size_t)nvf), skey(2 * (size_t)nvf), sval(2 * (size_t)nvf);
    KL(c, k_geo_pairs, nvf, f.agg.p, f.par1.p, nvf, nvc, key.p, val.p);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, key.p, skey.p, val.p, sval.p, 2 * nvf, 0, 32, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortPairs(A.temp(bytes), bytes, key.p, skey.p, val.p, sval.p, 2 * nvf, 0, 32, c.stream));
    f.agg_ptr.alloc((size_t)nvc + 1);
    KL(c, k_lower_bounds_i32, nvc + 1, skey.p, 2 * nvf, nvc, f.agg_ptr.p);
    int nvalid = 0;
    PNP_CUDA(cudaMemcpyAsync(&nvalid, f.agg_ptr.p + nvc, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    f.agg_mem.alloc(nvalid);
    PNP_CUDA(cudaMemcpyAsync(f.agg_mem.p, sval.p, (size_t)nvalid * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
    PNP_CUDA(cudaStreamSynchronize(c.stream));
  }
  auto nl = std::make_unique<Level>();
  nl->nv = nvc; nl->nslots = h.nslots; nl->rp = h.rp.p; nl->col = h.adj.p;
  nl->redisc = redisc;
  if (redisc) {
    nl->xy_own.alloc(nvc); nl->dmask_own.alloc(nvc);
    KL(c, k_level_geometry, nvc, h.int2ext.p, c.ext2int.p, c.xy.p, c.dmask.p, nvc, nl->xy_own.p, nl->dmask_own.p);
    nl->dm = nl->dmask_own.p;
    nl->u.fields = A.F; nl->u.d.alloc((size_t)A.F * nvc);
  } else { // Galerkin gather lists
    const long n4 = 4 * f.nslots;
    PNP_REQUIRE(n4 < (1l << 31) && f.nslots < (1l << 29), PNP_E_MESH, "multigrid: too many matrix slots on one level");
    DBuf<int> key(n4), skey(n4), err(1);
    DBuf<unsigned> val(n4), sval(n4);
    err.zero(c.stream);
    KL(c, k_geo_items, nvf, f.rp, f.col, nvf, f.agg.p, f.par1.p, nl->rp, nl->col, key.p, val.p, err.p);
    int herr = 0;
    err.download(&herr, 1, c.stream);
    PNP_REQUIRE(herr == 0, PNP_E_MESH, "multigrid: refinement levels are not nested");
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, key.p, skey.p, val.p, sval.p, (int)n4, 0, 32, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortPairs(A.temp(bytes), bytes, key.p, skey.p, val.p, sval.p, (int)n4, 0, 32, c.stream));
    key.release(); val.release();
    f.seg_ptr.alloc((size_t)nl->nslots + 1);
    KL(c, k_lower_bounds_i32, nl->nslots + 1, skey.p, (int)n4, (int)nl->nslots, f.seg_ptr.p);
    int nvalid = 0;
    PNP_CUDA(cudaMemcpyAsync(&nvalid, f.seg_ptr.p + nl->nslots, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    f.seg_items.alloc(nvalid); f.seg_w.alloc(nvalid);
    KL(c, k_geo_unpack, nvalid, sval.p, (long)nvalid, f.seg_items.p, f.seg_w.p);
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    c.launches += 4;
  }
  f.alpha = 1.0; // P1 interpolation needs no over-correction
  nl->vals_own.alloc((size_t)A.NP * nl->nslots);
  nl->vals = nl->vals_own.p;
  A.L.push_back(std::move(nl));
}

void alloc_work(Ctx& c, Amg& A, Level& l) {
  const size_t n = (size_t)A.F * l.nv, nall = (A.distributed && l.lc) ? (size_t)A.F * l.lc->nv : n;
  l.dinv.alloc(A.F == 3 ? 9 * (size_t)l.nv : n); l.x.alloc(nall); l.x2.alloc(nall); l.b.alloc(nall); l.r.alloc(nall);
  l.x.zero(c.stream); l.x2.zero(c.stream); l.b.zero(c.stream); l.r.zero(c.stream);
}

// distributed hierarchy: level li+1 lives on the child context `ref.lc`; transfers from the registered parent arrays
void coarsen_distributed(Ctx& c, Amg& A, int li, MgLevelRef& ref) {
  Level& f = *A.L[li];
  Ctx& fc = *f.lc; Ctx& kc = *ref.lc;
  const int nvf_all = (int)fc.nv, nvc = (int)kc.n_own;
  size_t bytes = 0;
  f.agg.alloc(nvf_all); f.par1.alloc(nvf_all);
  PNP_CUDA(cudaMemcpyAsync(f.agg.p, ref.par0.p, nvf_all * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
  PNP_CUDA(cudaMemcpyAsync(f.par1.p, ref.par1.p, nvf_all * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
  {
    DBuf<int> key(2 * (size_t)nvf_all), val(2 * (size_t)nvf_all), skey(2 * (size_t)nvf_all), sval(2 * (size_t)nvf_all);
    KL(c, k_geo_pairs, nvf_all, f.agg.p, f.par1.p, nvf_all, nvc, key.p, val.p);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, key.p, skey.p, val.p, sval.p, 2 * nvf_all, 0, 32, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortPairs(A.temp(bytes), bytes, key.p, skey.p, val.p, sval.p, 2 * nvf_all, 0, 32, c.stream));
    f.agg_ptr.alloc((size_t)nvc + 1);
    KL(c, k_lower_bounds_i32, nvc + 1, skey.p, 2 * nvf_all, nvc, f.agg_ptr.p);
    int nvalid = 0;
    PNP_CUDA(cudaMemcpyAsync(&nvalid, f.agg_ptr.p + nvc, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    f.agg_mem.alloc(nvalid);
    PNP_CUDA(cudaMemcpyAsync(f.agg_mem.p, sval.p, (size_t)nvalid * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
    PNP_CUDA(cudaStreamSynchronize(c.stream));
  }
  f.alpha = 1.0;
  auto nl = std::make_unique<Level>();
  nl->lc = &kc; nl->nv = nvc; nl->nslots = kc.nslots; nl->rp = kc.rp.p; nl->col = kc.adj.p;
  nl->dm = kc.dmask.p;
  nl->u.fields = A.F; nl->u.d.alloc((size_t)A.F * kc.nv); nl->u.d.zero(c.stream);
  nl->Amat.op = A.F == 3 ? OP_PNP : OP_PB; nl->Amat.nplanes = A.NP;
  nl->Amat.vals.alloc((size_t)A.NP * kc.nslots);
  nl->vals = nl->Amat.vals.p;
  A.L.push_back(std::move(nl));
}

void dense_factor(Ctx& c, Amg& A);

void dense_factor_global(Ctx& c, Amg& A);
void replica_setup(Ctx& c, Amg& A);

// matrix values of level li+1 from level li (one-GPU hierarchy): re-discretisation at the injected state for a `redisc`
// geometric level, else the Galerkin product P^T A P by deterministic gathers.  uf = state on level li (only followed
// through re-discretised levels); returns the state on level li+1.
const double* level_values(Ctx& c, Amg& A, int li, const double* uf, int comp0) {
  Level& l = *A.L[li]; Level& n = *A.L[li + 1];
  if (n.redisc) {
    if (A.F == 1) KL(c, k_inject<1>, l.nv, l.agg.p, l.par1.p, l.nv, uf, n.u.d.p);
    else KL(c, k_inject<3>, l.nv, l.agg.p, l.par1.p, l.nv, uf, n.u.d.p);
    c.acct(Ctx::ACC_TRANSFER, 8.0 * l.nv + 16.0 * A.F * n.nv);
    Operator op = c.last_op; op.aux0 = op.aux1 = -1;
    assemble_jacobian_on(c, StarView{n.rp, n.col, n.xy_own.p, n.dmask_own.p, n.nv}, n.nslots, op, n.u.d.p, n.vals_own.p,
                         A.NP, c.last_mode, c.last_eps);
    return n.u.d.p;
  }
  // constrained dofs of the finer level are left out of the product (only their unit diagonal has to be skipped)
  if (A.NP == 1)
    KL(c, k_galerkin<1>, n.nslots, l.seg_ptr.p, l.seg_items.p, l.seg_w.p, n.nslots, l.vals, l.nslots, n.vals_own.p, l.dm, l.col, l.rp, comp0);
  else if (A.NP == PNP_COMPACT_PLANES)
    KL(c, k_galerkin<PNP_COMPACT_PLANES>, n.nslots, l.seg_ptr.p, l.seg_items.p, l.seg_w.p, n.nslots, l.vals, l.nslots, n.vals_own.p, l.dm, l.col, l.rp, comp0);
  else
    KL(c, k_galerkin<7>, n.nslots, l.seg_ptr.p, l.seg_items.p, l.seg_w.p, n.nslots, l.vals, l.nslots, n.vals_own.p, l.dm, l.col, l.rp, comp0);
  c.acct(Ctx::ACC_ASSEMBLY, 8.0 * A.NP * ((double)l.nslots + (double)n.nslots) + 5.0 * (double)l.seg_items.n + 4.0 * (double)n.nslots);
  return nullptr;
}

// smoother matrix of level l (k_dinv): from the planes the level's cycle operations read
template <class T>
void level_dinv_t(Ctx& c, Amg& A, Level& l, const T* vals, long stride) {
  if (A.NP == 1) KL(c, (k_dinv<1, T>), l.nv, l.rp, vals, stride, l.nv, l.dinv.p);
  else if (A.NP == PNP_COMPACT_PLANES) KL(c, (k_dinv<PNP_COMPACT_PLANES, T>), l.nv, l.rp, vals, stride, l.nv, l.dinv.p);
  else KL(c, (k_dinv<7, T>), l.nv, l.rp, vals, stride, l.nv, l.dinv.p);
  c.acct(Ctx::ACC_ASSEMBLY, (4.0 + sizeof(T) * A.NP + (A.F == 3 ? 72.0 : 8.0)) * l.nv);
}
void level_dinv(Ctx& c, Amg& A, Level& l) {
  if (l.vals32.p) level_dinv_t<float>(c, A, l, l.vals32.p, l.stride32);
  else level_dinv_t<double>(c, A, l, l.vals, l.nslots);
}

// Which levels smooth against a single-precision companion of their matrix: one GPU (no partitioned or replicated
// hierarchy), damped Jacobi, a level the streaming SpMV serves, and at least mg_f32_min_rows rows (pnp_tune; -1: 2^22).
// The smoother and the residual of such a level read 4 bytes less per plane and slot (0.64x the bytes of a
// compact-layout pass); the multigrid is only a preconditioner, and the Krylov method keeps applying the fp64 matrix,
// so the accuracy a solve can reach is unchanged.  The default puts levels 7 and 6 of the pore mesh (47.1 M and 11.8 M
// vertices) on the float side; level 5 (2.9 M) and below, ~1 % of the step's bytes, stay in double, so that the
// cycle's corrections of the 5- and 7-plane layouts agree to rounding at those sizes.
bool mg_f32_rule(Ctx& c, const Amg& A, Level& l) {
  if (A.distributed || A.replica || A.smoother != 0) return false;
  const long t = tune().mg_f32_min_rows;
  if ((long)l.nv < (t >= 0 ? t : (1l << 22))) return false;
  StarOpArgs a{l.rp, l.col, l.vals, l.nslots, l.nv, l.x.p, l.x2.p};
  a.b = l.r.p;
  return star_op_tma_ok(c, a, EPI_JACOBI);
}
// (re)builds or drops level l's companion; true if the planes its cycle reads changed place
bool level_f32(Ctx& c, Amg& A, Level& l) {
  float* before = l.vals32.p;
  if (!mg_f32_rule(c, A, l)) { l.vals32.release(); l.stride32 = 0; return before != nullptr; }
  l.stride32 = (l.nslots + 3) & ~3l;
  const size_t n = (size_t)A.NP * l.stride32;
  if (l.vals32.n != n) l.vals32.alloc(n);
  const dim3 grid((unsigned)grid_for(l.stride32, BLK, 148 * 8), (unsigned)A.NP);
  k_round_planes<<<grid, BLK, 0, c.stream>>>(l.vals, l.nslots, l.nslots, l.vals32.p, l.stride32);
  PNP_CHECK_LAUNCH(); c.launches++;
  c.acct(Ctx::ACC_ASSEMBLY, (8.0 * l.nslots + 4.0 * l.stride32) * A.NP);
  return before != l.vals32.p;
}

// Gershgorin bounds of D^-1 A on every level (Chebyshev smoother); distributed: the maximum over the ranks
void gershgorin_bounds(Ctx& c, Amg& A) {
  DBuf<unsigned long long> d_l(A.L.size());
  d_l.zero(c.stream);
  for (size_t li = 0; li < A.L.size(); li++) {
    Level& l = *A.L[li];
    if (A.NP == 1) KL(c, k_gershgorin<1>, l.nv, l.rp, l.vals, l.nslots, l.nv, d_l.p + li);
    else if (A.NP == PNP_COMPACT_PLANES) KL(c, k_gershgorin<PNP_COMPACT_PLANES>, l.nv, l.rp, l.vals, l.nslots, l.nv, d_l.p + li);
    else KL(c, k_gershgorin<7>, l.nv, l.rp, l.vals, l.nslots, l.nv, d_l.p + li);
  }
  if (A.distributed) allreduce_max_u64(c, d_l.p, A.L.size());
  std::vector<unsigned long long> h = d_l.to_host(c.stream);
  for (size_t li = 0; li < A.L.size(); li++) {
    double v; std::memcpy(&v, &h[li], sizeof v);
    A.L[li]->lmax = (v > 0.0 && std::isfinite(v)) ? v : 2.0;
  }
}

void numeric(Ctx& c, Amg& A, int comp0) {
  if (A.distributed) {
    // re-discretise every coarser level at the injected state (what assemble_jacobian last linearised on the fine level)
    PNP_REQUIRE(c.last_u, PNP_E_ARG, "distributed multigrid needs the state of the last Jacobian assembly (the vector must stay alive)");
    PNP_REQUIRE(c.last_vals == A.L[0]->vals, PNP_E_ARG,
                "distributed multigrid re-discretises its coarse levels: the matrix must be the Jacobian of the last assembly");
    const double* uf = c.last_u;
    for (size_t li = 0; li + 1 < A.L.size(); li++) {
      Level& l = *A.L[li]; Level& n = *A.L[li + 1];
      const int nvf_all = (int)l.lc->nv;
      if (A.F == 1) KL(c, k_inject<1>, nvf_all, l.agg.p, l.par1.p, nvf_all, uf, n.u.d.p);
      else KL(c, k_inject<3>, nvf_all, l.agg.p, l.par1.p, nvf_all, uf, n.u.d.p);
      c.acct(Ctx::ACC_TRANSFER, 8.0 * nvf_all + 16.0 * A.F * n.nv);
      Operator op = c.last_op; op.aux0 = op.aux1 = -1;
      n.Amat.op = op.op;
      n.lc->launches = 0;
      assemble_jacobian(*n.lc, op, n.u, n.Amat, c.last_mode, c.last_eps); // (exchanges the ghost part of u first)
      c.absorb(*n.lc);
      uf = n.u.d.p;
    }
    for (size_t li = 0; li < A.L.size(); li++) level_dinv(c, A, *A.L[li]);
    if (c.mg_replica) replica_setup(c, A); else dense_factor_global(c, A);
    if (A.smoother == 1) gershgorin_bounds(c, A);
    return;
  }
  const double* uf = c.last_u;
  bool moved = false;
  for (size_t li = 0; li < A.L.size(); li++) {
    Level& l = *A.L[li];
    if (li + 1 < A.L.size()) uf = level_values(c, A, (int)li, uf, comp0);
    moved |= level_f32(c, A, l) && li > 0; // (level l's fp64 values are final here)
    level_dinv(c, A, l);
  }
  if (moved) A.cg_reset(); // the captured coarse correction names the planes its launches read
  A.dense_n = 0;
  if ((long)A.F * A.L.back()->nv <= A.dense_max) dense_factor(c, A); // (a one-level hierarchy is a direct solve)
  if (A.smoother == 1) gershgorin_bounds(c, A);
}

// ---- dense coarsest-level solve ----
template <int NP>
__global__ void k_dense_fill(const int* __restrict__ rp, const unsigned* __restrict__ col, const double* __restrict__ vals,
                             long stride, int nv, double* __restrict__ Ad, long n) {
  constexpr int F = NP == 1 ? 1 : 3;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < nv; r += gridDim.x * blockDim.x)
    for (int s = rp[r]; s < rp[r + 1]; s++) {
      const long cidx = col[s] & STAR_VMASK;
      if (cidx >= nv) continue;
      if (NP == 1) Ad[cidx * n + r] = vals[s];
      else {
        const PnpBlock B = pnp_block_at<NP>(vals, stride, s);
#pragma unroll
        for (int ki = 0; ki < 3; ki++)
#pragma unroll
          for (int kj = 0; kj < 3; kj++)
            if (pnp_plane(ki, kj) >= 0) Ad[(F * cidx + kj) * n + F * r + ki] = B.at(ki, kj);
      }
    }
}
__global__ void k_dense_fix_diag(double* __restrict__ Ad, long n) { // decoupled zero rows (all-Dirichlet coarse dofs)
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    if (Ad[i * n + i] == 0.0) Ad[i * n + i] = 1.0;
}
#define PNP_CUSOLVER(call)                                                                                          \
  do { cusolverStatus_t s_ = (call); if (s_ != CUSOLVER_STATUS_SUCCESS)                                             \
    throw ::pnp::Error(PNP_E_CUDA, std::string(#call) + " -> cusolver status " + std::to_string((int)s_)); } while (0)

void dense_factor(Ctx& c, Amg& A) {
  Level& l = *A.L.back();
  const long n = (long)A.F * l.nv;
  A.dense_n = (int)n;
  if (!A.cus) PNP_CUSOLVER(cusolverDnCreate(&A.cus));
  PNP_CUSOLVER(cusolverDnSetStream(A.cus, c.stream));
  if (A.dense.n != (size_t)(n * n)) { A.dense.alloc(n * n); A.dense_piv.alloc(n); A.dense_info.alloc(1); }
  A.dense.zero(c.stream);
  if (A.NP == 1) KL(c, k_dense_fill<1>, l.nv, l.rp, l.col, l.vals, l.nslots, l.nv, A.dense.p, n);
  else if (A.NP == PNP_COMPACT_PLANES) KL(c, k_dense_fill<PNP_COMPACT_PLANES>, l.nv, l.rp, l.col, l.vals, l.nslots, l.nv, A.dense.p, n);
  else KL(c, k_dense_fill<7>, l.nv, l.rp, l.col, l.vals, l.nslots, l.nv, A.dense.p, n);
  KL(c, k_dense_fix_diag, n, A.dense.p, n);
  int lwork = 0;
  PNP_CUSOLVER(cusolverDnDgetrf_bufferSize(A.cus, (int)n, (int)n, A.dense.p, (int)n, &lwork));
  if (A.dense_work.n < (size_t)lwork) A.dense_work.alloc(lwork);
  PNP_CUSOLVER(cusolverDnDgetrf(A.cus, (int)n, (int)n, A.dense.p, (int)n, A.dense_work.p, A.dense_piv.p, A.dense_info.p));
  c.acct(Ctx::ACC_DENSE, 24.0 * (double)n * (double)n); // zero fill + factor in place (read and write)
  int info = 0;
  A.dense_info.download(&info, 1, c.stream);
  PNP_REQUIRE(info == 0, PNP_E_BREAKDOWN, "multigrid: coarsest-level matrix is singular (LU info " + std::to_string(info) + ")");
}
void dense_solve(Ctx& c, Amg& A, Level& l) { // l.x = A^-1 l.b
  const long n = A.dense_n;
  PNP_CUDA(cudaMemcpyAsync(l.x.p, l.b.p, n * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
  PNP_CUSOLVER(cusolverDnDgetrs(A.cus, CUBLAS_OP_N, (int)n, 1, A.dense.p, (int)n, A.dense_piv.p, l.x.p, (int)n, A.dense_info.p));
  c.launches += 2; c.acct(Ctx::ACC_DENSE, 8.0 * (double)n * (double)n);
}

// coarsest level of the distributed hierarchy: every rank contributes its owned rows, the matrix is summed over the
// ranks and factorised redundantly; each cycle sums the right-hand side the same way
void dense_factor_global(Ctx& c, Amg& A) {
  Level& l = *A.L.back();
  const long n = (long)A.F * c.mg_nglobal;
  A.dense_n = (int)n;
  if (!A.cus) PNP_CUSOLVER(cusolverDnCreate(&A.cus));
  PNP_CUSOLVER(cusolverDnSetStream(A.cus, c.stream));
  if (A.dense.n != (size_t)(n * n)) { A.dense.alloc(n * n); A.dense_piv.alloc(n); A.dense_info.alloc(1); A.grhs.alloc(n); }
  A.dense.zero(c.stream);
  const unsigned char* dm = c.mg_aggregated ? l.lc->dmask.p : nullptr;
  if (A.NP == 1) KL(c, k_dense_fill_global<1>, l.nv, l.rp, l.col, l.vals, l.nslots, l.nv, c.mg_gid.p, A.dense.p, n, dm, A.comp0);
  else if (A.NP == PNP_COMPACT_PLANES)
    KL(c, k_dense_fill_global<PNP_COMPACT_PLANES>, l.nv, l.rp, l.col, l.vals, l.nslots, l.nv, c.mg_gid.p, A.dense.p, n, dm, A.comp0);
  else KL(c, k_dense_fill_global<7>, l.nv, l.rp, l.col, l.vals, l.nslots, l.nv, c.mg_gid.p, A.dense.p, n, dm, A.comp0);
  allreduce_sum(c, A.dense.p, (size_t)(n * n));
  KL(c, k_dense_fix_diag, n, A.dense.p, n);
  int lwork = 0;
  PNP_CUSOLVER(cusolverDnDgetrf_bufferSize(A.cus, (int)n, (int)n, A.dense.p, (int)n, &lwork));
  if (A.dense_work.n < (size_t)lwork) A.dense_work.alloc(lwork);
  static const bool timing = std::getenv("PNP_AMG_TIMING") != nullptr;
  if (timing) PNP_CUDA(cudaStreamSynchronize(c.stream));
  const auto t0 = std::chrono::steady_clock::now();
  PNP_CUSOLVER(cusolverDnDgetrf(A.cus, (int)n, (int)n, A.dense.p, (int)n, A.dense_work.p, A.dense_piv.p, A.dense_info.p));
  int info = 0;
  A.dense_info.download(&info, 1, c.stream);
  if (timing) std::printf("[amg] rank %d global dense LU n = %ld: %.1f ms\n", c.rank, n,
                          1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
  PNP_REQUIRE(info == 0, PNP_E_BREAKDOWN, "multigrid: coarsest-level matrix is singular (LU info " + std::to_string(info) + ")");
}
// aggregated variant: the coarsest distributed level was smoothed; its residual (l.r) is summed per aggregate over all
// ranks, the dense aggregate system is solved redundantly and the correction is added back (piecewise constant)
void dense_correct_aggregated(Ctx& c, Amg& A, Level& l) {
  const long n = A.dense_n;
  A.grhs.zero(c.stream);
  if (A.F == 1) KL(c, k_to_global<1>, l.nv, l.r.p, c.mg_gid.p, l.nv, A.grhs.p);
  else KL(c, k_to_global<3>, l.nv, l.r.p, c.mg_gid.p, l.nv, A.grhs.p);
  allreduce_sum(c, A.grhs.p, (size_t)n);
  PNP_CUSOLVER(cusolverDnDgetrs(A.cus, CUBLAS_OP_N, (int)n, 1, A.dense.p, (int)n, A.dense_piv.p, A.grhs.p, (int)n, A.dense_info.p));
  if (A.F == 1) KL(c, k_add_from_global<1>, l.nv, A.grhs.p, c.mg_gid.p, l.nv, A.alpha, l.x.p, l.lc->dmask.p, A.comp0);
  else KL(c, k_add_from_global<3>, l.nv, A.grhs.p, c.mg_gid.p, l.nv, A.alpha, l.x.p, l.lc->dmask.p, A.comp0);
  c.launches += 2;
}
void dense_solve_global(Ctx& c, Amg& A, Level& l) {
  const long n = A.dense_n;
  A.grhs.zero(c.stream);
  if (A.F == 1) KL(c, k_to_global<1>, l.nv, l.b.p, c.mg_gid.p, l.nv, A.grhs.p);
  else KL(c, k_to_global<3>, l.nv, l.b.p, c.mg_gid.p, l.nv, A.grhs.p);
  allreduce_sum(c, A.grhs.p, (size_t)n);
  PNP_CUSOLVER(cusolverDnDgetrs(A.cus, CUBLAS_OP_N, (int)n, 1, A.dense.p, (int)n, A.dense_piv.p, A.grhs.p, (int)n, A.dense_info.p));
  const int nloc = (int)l.lc->nv; // owned and ghost vertices: no halo exchange needed afterwards
  if (A.F == 1) KL(c, k_from_global<1>, nloc, A.grhs.p, c.mg_gid.p, nloc, l.x.p);
  else KL(c, k_from_global<3>, nloc, A.grhs.p, c.mg_gid.p, nloc, l.x.p);
  c.launches += 2;
}

} // namespace
void amg_setup(Ctx& c, Solver& S, const Matrix& M);
void amg_apply(Ctx& c, Solver& S, const Matrix&, const double* d, double* y);
namespace {
// replica variant of the coarsest distributed level.  Numeric setup: the injected state of that level is summed to the
// replica (every vertex is owned by exactly one rank), the replica re-discretises its operator and sets up its own
// hierarchy.  Solve: gather the right-hand side, one cycle of the replica's multigrid, scatter to owned + ghost vertices.
void replica_setup(Ctx& c, Amg& A) {
  Ctx& rc = *c.mg_replica;
  Level& l = *A.L.back();
  const long n = (long)A.F * c.mg_nglobal;
  A.dense_n = (int)n; // marks the coarsest level as "solved below"
  if (A.grhs.n != (size_t)n) { A.grhs.alloc(n); A.rep_x.alloc(n); A.rep_u.d.alloc(n); }
  A.rep_u.fields = A.F;
  A.rep_u.d.zero(c.stream);
  if (A.F == 1) KL(c, k_to_global<1>, l.nv, l.u.d.p, c.mg_gid.p, l.nv, A.rep_u.d.p);
  else KL(c, k_to_global<3>, l.nv, l.u.d.p, c.mg_gid.p, l.nv, A.rep_u.d.p);
  allreduce_sum(c, A.rep_u.d.p, (size_t)n);
  Operator op = c.last_op; op.aux0 = op.aux1 = -1;
  A.rep_A.op = op.op; A.rep_A.nplanes = A.NP;
  if (A.rep_A.vals.n != (size_t)A.NP * rc.nslots) A.rep_A.vals.alloc((size_t)A.NP * rc.nslots);
  rc.launches = 0;
  assemble_jacobian(rc, op, A.rep_u, A.rep_A, c.last_mode, c.last_eps);
  if (!A.rep_solver) {
    A.rep_solver = std::make_unique<Solver>(); A.rep_solver->prec = PNP_PREC_AMG;
    A.rep_solver->amg = std::make_shared<Amg>(); A.rep_solver->amg->replica = true;
  }
  auto& ro = A.rep_solver->opts;
  ro["amg_geometric"] = 1; /* refinement levels the replica made itself, if any */ ro["amg_omega"] = A.omega; ro["amg_alpha"] = A.alpha; ro["amg_gamma"] = A.gamma;
  ro["amg_dense_max"] = A.dense_max; ro["amg_coarse_sweeps"] = A.coarse_sweeps; ro["amg_smoother"] = A.smoother;
  ro["amg_cheb_ratio"] = A.cheb_ratio; ro["amg_pre_steps"] = A.pre_steps; ro["amg_post_steps"] = A.post_steps;
  amg_setup(rc, *A.rep_solver, A.rep_A);
  c.absorb(rc);
}
void replica_solve(Ctx& c, Amg& A, Level& l, int nu) {
  Ctx& rc = *c.mg_replica;
  const long n = (long)A.F * c.mg_nglobal;
  A.grhs.zero(c.stream);
  if (A.F == 1) KL(c, k_to_global<1>, l.nv, l.b.p, c.mg_gid.p, l.nv, A.grhs.p);
  else KL(c, k_to_global<3>, l.nv, l.b.p, c.mg_gid.p, l.nv, A.grhs.p);
  allreduce_sum(c, A.grhs.p, (size_t)n);
  A.rep_solver->prec_steps = nu;
  rc.launches = 0;
  amg_apply(rc, *A.rep_solver, A.rep_A, A.grhs.p, A.rep_x.p);
  const int nloc = (int)l.lc->nv; // owned and ghost vertices: no halo exchange needed afterwards
  if (A.F == 1) KL(c, k_from_global<1>, nloc, A.rep_x.p, c.mg_gid.p, nloc, l.x.p);
  else KL(c, k_from_global<3>, nloc, A.rep_x.p, c.mg_gid.p, nloc, l.x.p);
  c.absorb(rc); c.launches += 2;
}

void jacobi0(Ctx& c, Amg& A, Level& l, double omega, double* dvec) {
  if (A.F == 1) KL(c, k_jacobi0<1>, l.nv, l.dinv.p, l.b.p, omega, l.x.p, l.nv, dvec);
  else KL(c, k_jacobi0<3>, l.nv, l.dinv.p, l.b.p, omega, l.x.p, l.nv, dvec);
  c.acct(Ctx::ACC_TRANSFER, ((A.F == 3 ? 72.0 : 8.0) + 16.0 * A.F + (dvec ? 8.0 * A.F : 0.0)) * l.nv);
}

// `steps` smoothing steps on level l for A x = b; zero: x starts from 0.  Result in l.x.
void smooth(Ctx& c, Amg& A, Level& l, int steps, bool zero) {
  const long n = (long)A.F * l.nv;
  if (steps <= 0) { if (zero) PNP_CUDA(cudaMemsetAsync(l.x.p, 0, n * sizeof(double), c.stream)); return; }
  if (A.smoother == 0) {
    int s = 0;
    if (zero) { jacobi0(c, A, l, A.omega, nullptr); s = 1; }
    for (; s < steps; s++) { level_op<2>(c, A, l, l.x.p, l.b.p, l.x2.p); std::swap(l.x.p, l.x2.p); }
    return;
  }
  if (A.smoother == 2) {
    // SeqSSOR(w = 1) as ISTL's AMG applies it (ISTLBackend_NOVLP_CG_AMG_SSOR, instationary_pnp_from_pb_md.hh:208-211): a step is a
    // forward and a backward Gauss-Seidel sweep over the level's rows, in place; the finest level sweeps in the reference's
    // row order (the order of the SSOR preconditioner), the coarser ones in their own.  Level-scheduled like pnp_precond.cu.
    const bool finest = &l == A.L[0].get();
    const SweepView V{l.rp, l.col, finest ? c.int2ext.p : nullptr, l.nv};
    if (!l.gs_plan) l.gs_plan = sweep_plan_build(c, V, A.F);
    if (zero) PNP_CUDA(cudaMemsetAsync(l.x.p, 0, n * sizeof(double), c.stream));
    for (int s = 0; s < steps; s++) {
      sweep_gs(c, *l.gs_plan, V, l.vals, l.nslots, l.b.p, l.x.p, +1);
      sweep_gs(c, *l.gs_plan, V, l.vals, l.nslots, l.b.p, l.x.p, -1);
    }
    c.acct(finest ? Ctx::ACC_SPMV_FINE : Ctx::ACC_SPMV_COARSE, 2.0 * steps * ((8.0 * A.NP + 4.0) * (double)l.nslots + 24.0 * n));
    return;
  }
  // Chebyshev polynomial smoother for D^-1 A on [lmax/ratio, 1.1*lmax]; l.r holds the direction d
  const double lmx = 1.1 * l.lmax, lmn = l.lmax / A.cheb_ratio;
  const double theta = 0.5 * (lmx + lmn), delta = 0.5 * (lmx - lmn), sigma = theta / delta;
  double rho = 1.0 / sigma;
  int s = 0;
  if (zero) { jacobi0(c, A, l, 1.0 / theta, l.r.p); s = 1; }
  else { level_op<3>(c, A, l, l.x.p, l.b.p, l.x2.p, 1.0 / theta, 0.0, l.r.p); std::swap(l.x.p, l.x2.p); s = 1; }
  for (; s < steps; s++) {
    const double rho_new = 1.0 / (2.0 * sigma - rho);
    level_op<3>(c, A, l, l.x.p, l.b.p, l.x2.p, 2.0 * rho_new / delta, rho_new * rho, l.r.p);
    std::swap(l.x.p, l.x2.p);
    rho = rho_new;
  }
}

void cycle(Ctx& c, Amg& A, int li, int nu, int comp0, bool zero);

// The part of one cycle below the finest level (right-hand side in L[1]->b, result in L[1]->x), replayed from a CUDA graph
void coarse_correction(Ctx& c, Amg& A, int nu, int comp0) {
  auto direct = [&] {
    const int visits = 0 < A.wlevels ? A.gamma : 1;
    for (int g = 0; g < visits; g++) cycle(c, A, 1, nu, comp0, g == 0);
  };
  auto snapshot = [&](std::vector<std::pair<double*, double*>>& v) {
    v.clear();
    for (size_t li = 1; li < A.L.size(); li++) v.push_back({A.L[li]->x.p, A.L[li]->x2.p});
  };
  auto restore = [&](const std::vector<std::pair<double*, double*>>& v) {
    for (size_t li = 1; li < A.L.size(); li++) { A.L[li]->x.p = v[li - 1].first; A.L[li]->x2.p = v[li - 1].second; }
  };
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  PNP_CUDA(cudaStreamIsCapturing(c.stream, &cap));
  // (Chebyshev coefficients change with every numeric set-up; a replica's cycle runs inside its parent's capture)
  if (!tune().graph || A.cg_failed || A.smoother != 0 || cap != cudaStreamCaptureStatusNone) { direct(); return; }
  const double key[8] = {(double)nu, A.omega, (double)A.gamma, (double)A.wlevels, (double)A.pre_steps, (double)A.post_steps,
                         (double)A.coarse_sweeps, (double)comp0 + 16.0 * A.dense_n};
  if (A.cg_exec && std::memcmp(key, A.cg_key, sizeof key) != 0) A.cg_reset();
  if (!A.cg_exec) {
    if (A.cg_calls++ < 1) { direct(); return; } // first application: plain launches (libraries set up their work space)
    std::memcpy(A.cg_key, key, sizeof key);
    snapshot(A.cg_before);
    const long l0 = c.launches;
    double b0[Ctx::ACC_N];
    for (int k = 0; k < Ctx::ACC_N; k++) b0[k] = c.alg_bytes[k];
    cudaGraph_t graph = nullptr;
    bool ok = cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
      try { direct(); } catch (const Error&) { ok = false; }
      if (cudaStreamEndCapture(c.stream, &graph) != cudaSuccess || !graph) ok = false;
    }
    if (ok && cudaGraphInstantiate(&A.cg_exec, graph, 0) != cudaSuccess) { ok = false; A.cg_exec = nullptr; }
    if (graph) cudaGraphDestroy(graph);
    A.cg_launches = c.launches - l0; c.launches = l0;               // (nothing has run yet)
    for (int k = 0; k < Ctx::ACC_N; k++) { A.cg_bytes[k] = c.alg_bytes[k] - b0[k]; c.alg_bytes[k] = b0[k]; }
    snapshot(A.cg_after);
    if (!ok) { // capture not possible here (a library call that cannot be captured): plain launches from now on
      cudaGetLastError();
      A.cg_failed = true; A.cg_exec = nullptr;
      restore(A.cg_before);
      direct();
      return;
    }
  }
  restore(A.cg_before);
  PNP_CUDA(cudaGraphLaunch(A.cg_exec, c.stream));
  restore(A.cg_after);
  c.launches += A.cg_launches;
  for (int k = 0; k < Ctx::ACC_N; k++) c.alg_bytes[k] += A.cg_bytes[k];
}

// one multigrid cycle on level li for A x = b (gamma = 1: V, 2: W); zero: x starts from 0.  Result in l.x
void cycle(Ctx& c, Amg& A, int li, int nu, int comp0, bool zero) {
  Level& l = *A.L[li];
  const bool coarsest = li + 1 == (int)A.L.size();
  if (coarsest && A.dense_n > 0 && A.distributed && c.mg_aggregated) { // smoothed level on top of the replicated aggregate solve
    smooth(c, A, l, nu, zero);
    level_op<1>(c, A, l, l.x.p, l.b.p, l.r.p);
    dense_correct_aggregated(c, A, l);
    smooth(c, A, l, nu, false);
    return;
  }
  if (coarsest && A.dense_n > 0) {
    if (A.distributed && c.mg_replica) replica_solve(c, A, l, nu);
    else if (A.distributed) dense_solve_global(c, A, l);
    else dense_solve(c, A, l);
    return;
  }
  const int nu_pre = A.pre_steps >= 0 ? A.pre_steps : nu, nu_post = A.post_steps >= 0 ? A.post_steps : nu;
  smooth(c, A, l, coarsest ? A.coarse_sweeps : nu_pre, zero);
  if (coarsest) return;
  Level& nx = *A.L[li + 1];
  level_op<1>(c, A, l, l.x.p, l.b.p, l.r.p);
  if (A.distributed) halo_exchange(*l.lc, l.r.p, A.F); // children of an owned coarse vertex may be ghosts here
  if (A.F == 1) KL(c, k_restrict<1>, nx.nv, l.agg_ptr.p, l.agg_mem.p, l.par1.p, nx.nv, l.r.p, nx.b.p);
  else KL(c, k_restrict<3>, nx.nv, l.agg_ptr.p, l.agg_mem.p, l.par1.p, nx.nv, l.r.p, nx.b.p);
  c.acct(Ctx::ACC_TRANSFER, (8.0 * A.F + 4.0) * l.nv + 4.0 * (double)l.agg_mem.n + (8.0 * A.F + 4.0) * nx.nv);
  if (nx.dm) { // re-discretised coarse levels carry their own Dirichlet rows: no residual into them
    if (A.F == 1) KL(c, k_mask_dirichlet<1>, nx.nv, nx.b.p, nx.dm, nx.nv, comp0);
    else KL(c, k_mask_dirichlet<3>, nx.nv, nx.b.p, nx.dm, nx.nv, comp0);
    c.acct(Ctx::ACC_TRANSFER, 1.0 * nx.nv);
  }
  if (li == 0) coarse_correction(c, A, nu, comp0);
  else {
    const int visits = li < A.wlevels ? A.gamma : 1;
    for (int g = 0; g < visits; g++) cycle(c, A, li + 1, nu, comp0, g == 0);
  }
  if (A.distributed && !(li + 2 == (int)A.L.size() && A.dense_n > 0 && !c.mg_aggregated)) halo_exchange(*nx.lc, nx.x.p, A.F); // parents may be ghosts
  const unsigned char* dm = l.dm; // constrained dofs of this level receive no correction
  if (A.F == 1) KL(c, k_prolong<1>, l.nv, l.agg.p, l.par1.p, l.nv, nx.x.p, l.alpha, l.x.p, dm, comp0);
  else KL(c, k_prolong<3>, l.nv, l.agg.p, l.par1.p, l.nv, nx.x.p, l.alpha, l.x.p, dm, comp0);
  c.acct(Ctx::ACC_TRANSFER, (16.0 * A.F + 9.0) * l.nv + 8.0 * A.F * nx.nv);
  smooth(c, A, l, nu_post, false);
}

} // namespace

// 1: the coarse correction is replayed from a CUDA graph, -1: capture failed (plain launches), 0: not captured (yet)
int amg_graph_state(const Solver& S) { return !S.amg ? 0 : (S.amg->cg_exec ? 1 : (S.amg->cg_failed ? -1 : 0)); }

void amg_setup(Ctx& c, Solver& S, const Matrix& M) {
  if (!S.amg) S.amg = std::make_shared<Amg>();
  Amg& A = *S.amg;
  const int comp0 = M.comp0;
  A.comp0 = comp0;
  // one GPU with refinement levels: re-discretise the coarse operators (cheaper than the Galerkin gathers by an order of
  // magnitude, and what the distributed hierarchy does) when M is the plain Jacobian of the last assembly
  const bool want_redisc = S.opt("amg_geometric", 1) != 0 && S.opt("amg_rediscretise", 1) != 0 && c.n_own == c.nv &&
                           !c.hier.empty() && c.mg.empty() && c.last_u && c.last_vals == M.vals.p &&
                           (M.op == OP_PB || M.op == OP_PNP || M.op == OP_MASS);
  const double sym_key = S.opt("amg_geometric", 1) + 3.0 * S.opt("amg_dense_max", 4096) + 1e7 * S.opt("amg_alpha", 1.6);
  if (!A.symbolic || A.NP != M.nplanes || A.nv0 != c.n_own || A.nslots0 != c.nslots || A.redisc != want_redisc ||
      A.mg_epoch != c.mg_epoch || A.sym_key != sym_key) {
    A.L.clear(); A.cg_reset(); A.cg_failed = false;
    A.NP = M.nplanes; A.F = M.nplanes == 1 ? 1 : 3;
    A.nv0 = c.n_own; A.nslots0 = c.nslots; A.mg_epoch = c.mg_epoch; A.sym_key = sym_key;
    auto l0 = std::make_unique<Level>();
    l0->nv = (int)c.n_own; l0->nslots = c.nslots; l0->rp = c.rp.p; l0->col = c.adj.p; l0->vals = M.vals.p;
    A.L.push_back(std::move(l0));
    A.alpha = S.opt("amg_alpha", 1.6);
    A.L[0]->lc = &c;
    A.L[0]->dm = c.dmask.p;
    A.redisc = want_redisc;
    A.distributed = S.opt("amg_geometric", 1) != 0 && !c.mg.empty() && c.mg_nglobal > 0 &&
                    (M.op == OP_PB || M.op == OP_PNP || M.op == OP_MASS);
    if (A.distributed) {
      for (auto& ref : c.mg) coarsen_distributed(c, A, (int)A.L.size() - 1, ref);
      A.n_geo = (int)c.mg.size();
    }
    // geometric levels: every coarser level of the refinement hierarchy (if the mesh was refined in this context)
    const bool geometric = !A.distributed && S.opt("amg_geometric", 1) != 0 && c.n_own == c.nv && !c.hier.empty();
    if (!A.distributed) A.n_geo = 0;
    if (geometric) {
      const int* i2e = c.int2ext.p;
      const double* uf = c.last_u;
      for (int hi = (int)c.hier.size() - 1; hi >= 0; hi--) {
        const int li = (int)A.L.size() - 1;
        coarsen_geometric(c, A, li, c.hier[hi], i2e, A.redisc);
        i2e = c.hier[hi].int2ext.p;
        uf = level_values(c, A, li, uf, comp0); // the aggregation below needs the numeric values
        A.n_geo++;
      }
    }
    // algebraic levels below: aggregates from the strength of connection of the current matrix values, level by level
    A.dense_max = (int)S.opt("amg_dense_max", 4096);
    for (int li = (int)A.L.size() - 1; li < 24 && !A.distributed; li++) {
      if (A.L[li]->nv <= 64 || (long)A.F * A.L[li]->nv <= A.dense_max) break;
      if (!coarsen(c, A, li)) break;
      // numeric values of the new level are needed before it can be coarsened further
      level_values(c, A, li, nullptr, comp0);
    }
    for (auto& l : A.L) alloc_work(c, A, *l);
    if (!A.distributed) { // level 0 iterates are SpMV inputs whose ghost columns must read as zero
      Level& l0r = *A.L[0];
      const size_t nall = (size_t)A.F * c.nv;
      l0r.x.alloc(nall); l0r.x2.alloc(nall);
      l0r.x.zero(c.stream); l0r.x2.zero(c.stream);
    }
    A.symbolic = true;
    if (S.verbosity > 0) {
      std::printf("multigrid hierarchy (%d geometric transfers):", A.n_geo);
      for (auto& l : A.L) std::printf(" %d", l->nv);
      std::printf("\n");
    }
  }
  A.L[0]->vals = M.vals.p;
  static const bool timing = std::getenv("PNP_AMG_TIMING") != nullptr;
  if (timing) PNP_CUDA(cudaStreamSynchronize(c.stream));
  const auto t_num0 = std::chrono::steady_clock::now();
  A.omega = S.opt("amg_omega", 0.7); A.gamma = (int)S.opt("amg_gamma", 1); A.wlevels = (int)S.opt("amg_wlevels", 99);
  A.coarse_sweeps = (int)S.opt("amg_coarse_sweeps", 40); A.smoother = (int)S.opt("amg_smoother", 0);
  PNP_REQUIRE(A.smoother >= 0 && A.smoother <= 2, PNP_E_ARG, "amg_smoother: 0 damped Jacobi, 1 Chebyshev, 2 symmetric Gauss-Seidel");
  PNP_REQUIRE(A.smoother != 2 || !A.distributed, PNP_E_ARG, "the Gauss-Seidel smoother sweeps the rows of one GPU: use Jacobi / Chebyshev on a partitioned mesh");
  PNP_REQUIRE(A.smoother != 2 || A.NP != PNP_COMPACT_PLANES, PNP_E_ARG, "the Gauss-Seidel smoother sweeps 7-plane PNP matrices only");
  A.cheb_ratio = S.opt("amg_cheb_ratio", 8.0);
  A.pre_steps = (int)S.opt("amg_pre_steps", -1); A.post_steps = (int)S.opt("amg_post_steps", -1);
  numeric(c, A, comp0);
  if (timing) {
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    std::printf("[amg] rank %d numeric setup %.1f ms (levels %zu, dense n = %d, distributed %d)\n", c.rank,
                1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t_num0).count(), A.L.size(), A.dense_n,
                (int)A.distributed);
  }
}

// y = M^{-1} d : `prec_steps` pre- and post-smoothing sweeps per level
void amg_apply(Ctx& c, Solver& S, const Matrix&, const double* d, double* y) {
  Amg& A = *S.amg;
  Level& l0 = *A.L[0];
  const long n = (long)A.F * l0.nv;
  const int nu = S.prec_steps > 0 ? S.prec_steps : 1;
  if (c.n_own == c.nv) {
    // one GPU: the finest level works on the caller's vectors -- d is its right-hand side and y one of its two iterate
    // buffers.  A cycle swaps the iterate buffers (pre - 1) + post times (the first pre-smoothing step starts from zero
    // and writes in place); y starts as the spare buffer if that count is odd, as the iterate if it is even, so the
    // result lands in y: no vector copies around the cycle (2 x 2.3 GB of traffic per application at k = 7).
    double *keep_b = l0.b.p, *keep_x = l0.x.p, *keep_x2 = l0.x2.p;
    const int pre = A.pre_steps >= 0 ? A.pre_steps : nu, post = A.post_steps >= 0 ? A.post_steps : nu;
    const int swaps = A.smoother == 2 ? 0 : (pre > 0 ? pre - 1 : 0) + post; // (Gauss-Seidel sweeps work in place)
    struct Restore { // the level's buffers own their memory: put the pointers back whatever happens in the cycle
      Level& l; double *b, *x, *x2;
      ~Restore() { l.b.p = b; l.x.p = x; l.x2.p = x2; }
    } restore{l0, keep_b, keep_x, keep_x2};
    l0.b.p = const_cast<double*>(d);
    if (swaps & 1) l0.x2.p = y; else l0.x.p = y;
    cycle(c, A, 0, nu, A.comp0, true);
    double* result = l0.x.p;
    if (result != y) { PNP_CUDA(cudaMemcpyAsync(y, result, n * sizeof(double), cudaMemcpyDeviceToDevice, c.stream)); c.acct(Ctx::ACC_BLAS1, 16.0 * n); }
    return;
  }
  PNP_CUDA(cudaMemcpyAsync(l0.b.p, d, n * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
  cycle(c, A, 0, nu, A.comp0, true);
  PNP_CUDA(cudaMemcpyAsync(y, l0.x.p, n * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
}

} // namespace pnp
