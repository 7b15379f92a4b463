// pnp_precond.cu -- SSOR(k) and ILU0 preconditioners with the reference's sequential sweep semantics.
//
// Replaces ISTL's SeqSSOR / SeqILU0 inside PDELab's ISTLBackend_NOVLP_BCGS_SSORk (the reference's default backend,
// /root/reference/src/instationary_pnp_from_pb_md.hh:188-191; SURVEY App. A.7-A.8).  Both sweep the dofs in matrix-row
// order; the device runs the SAME sweep by level scheduling (pnp_sweep.cuh): the dofs are grouped into levels of mutually
// uncoupled dofs in the reference's order, one launch per large level, runs of small levels inside one single-block
// kernel (block barrier between levels).  Results equal the sequential sweep up to the summation order inside a row,
// so Krylov iteration counts match the CPU path.  With several ranks the sweeps act on the local diagonal block
// (ghost columns skipped), like the NOVLP backends.
//
// Cost: the number of levels is the longest chain of coupled dofs in the reference's numbering: 18-100 on the Gmsh meshes,
// 10-35 on refined ones (old vertices are numbered before the edge midpoints, which keeps the chains short), so a sweep
// is one matrix pass in a few dozen launches at any size.  They are the parity preconditioners because their Krylov
// iteration counts grow like 1/h; the multigrid of pnp_amg.cu is the fast one.
// HBM traffic per sweep = one pass over the matrix planes (8*NP*nslots) + adjacency (4*nslots per field) + vectors.
#include <cub/cub.cuh>

#include "pnp_common.cuh"
#include "pnp_sweep.cuh"

namespace pnp {

struct SweepSegment { int l0, l1; bool single_block; }; // levels [l0, l1)
struct SweepPlan {
  int F = 1; bool full = false; int nlev = 0; long n = 0;
  DBuf<int> dofs;              // dof ids (F*v + f) sorted by level
  DBuf<int> d_lptr;            // device copy of lptr
  std::vector<int> lptr;       // nlev + 1
  std::vector<SweepSegment> seg;
};
struct SweepPrec {
  std::shared_ptr<SweepPlan> plan_ssor, plan_ilu;
  DBuf<double> lu;             // ILU0 factor: F*F planes of nslots
};

namespace {

constexpr int SB_THREADS = 1024;   // single-block kernel
constexpr int SB_MAX_LEVEL = 4096; // levels up to this many dofs may share a single-block launch

enum : int { FN_GS = 0, FN_ILU_FACTOR = 1, FN_ILU_FWD = 2, FN_ILU_BWD = 3 };
struct SweepArgs {
  SweepView S; const double* vals; double* lu; long stride; const double* d; double* x;
};
template <int F, int FN> __device__ __forceinline__ void sweep_item(const SweepArgs& a, int dof) {
  const int v = dof / F, f = dof - F * v;
  if (FN == FN_GS) gs_update<(F == 1 ? 1 : 7)>(a.S, a.vals, a.stride, a.d, a.x, v, f);
  else if (FN == FN_ILU_FACTOR) ilu0_row<F>(a.S, a.lu, a.stride, v, f);
  else if (FN == FN_ILU_FWD) ilu0_forward<F>(a.S, a.lu, a.stride, a.d, a.x, v, f);
  else ilu0_backward<F>(a.S, a.lu, a.stride, a.x, v, f);
}
// one level, many blocks
template <int F, int FN> __global__ void __launch_bounds__(256) k_sweep_level(const SweepArgs a, const int* __restrict__ dofs,
                                                                              int begin, int end) {
  for (int i = begin + blockIdx.x * blockDim.x + threadIdx.x; i < end; i += gridDim.x * blockDim.x) sweep_item<F, FN>(a, dofs[i]);
}
// levels l0 .. l1-1 (dir = +1) or l1-1 .. l0 (dir = -1) in ONE block, block barrier between levels
template <int F, int FN> __global__ void __launch_bounds__(SB_THREADS) k_sweep_levels(const SweepArgs a, const int* __restrict__ dofs,
                                                                                      const int* __restrict__ lptr, int l0, int l1, int dir) {
  for (int k = 0; k < l1 - l0; k++) {
    const int l = dir > 0 ? l0 + k : l1 - 1 - k;
    const int b = lptr[l], e = lptr[l + 1];
    for (int i = b + threadIdx.x; i < e; i += blockDim.x) sweep_item<F, FN>(a, dofs[i]);
    __syncthreads();
  }
}

template <int F> __global__ void k_level_relax(const SweepView S, int* lev, bool full, int* changed) {
  for (int dof = blockIdx.x * blockDim.x + threadIdx.x; dof < F * S.n_own; dof += gridDim.x * blockDim.x) {
    const int v = dof / F, f = dof - F * v;
    // in-place (asynchronous) relaxation: values only grow and never pass the true level, the fixpoint is the level
    const int l = sweep_level_relax<F>(S, lev, v, f, full);
    if (l != lev[dof]) { lev[dof] = l; *changed = 1; }
  }
}
__global__ void k_iota_int(int* a, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) a[i] = i;
}
__global__ void k_level_starts(const int* __restrict__ sorted_lev, int n, int nlev, int* __restrict__ lptr) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (i == 0 || sorted_lev[i] != sorted_lev[i - 1]) lptr[sorted_lev[i]] = i;
    if (i == n - 1) lptr[nlev] = n;
  }
}
// 7 stored planes -> the 9 blocks of PDELab's pattern (ILU0 fills the (c+,c-) / (c-,c+) blocks)
__global__ void k_planes_7_to_9(const double* __restrict__ vals, long stride, double* __restrict__ lu) {
  for (long s = blockIdx.x * (long)blockDim.x + threadIdx.x; s < stride; s += (long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int f = 0; f < 3; f++)
#pragma unroll
      for (int g = 0; g < 3; g++) {
        const int pl = pnp_plane7(f, g);
        lu[(long)(3 * f + g) * stride + s] = pl >= 0 ? vals[(long)pl * stride + s] : 0.0;
      }
  }
}

SweepView view_of(const Ctx& c) { return SweepView{c.rp.p, c.adj.p, c.int2ext.p, (int)c.n_own}; }

std::shared_ptr<SweepPlan> build_plan_view(Ctx& c, const SweepView& S, int F, bool full) {
  auto P = std::make_shared<SweepPlan>();
  P->F = F; P->full = full; P->n = (long)F * S.n_own;
  const int n = (int)P->n;
  PNP_REQUIRE(P->n < (1l << 31), PNP_E_MESH, "too many dofs for a level-scheduled sweep");
  DBuf<int> lev(n), changed(1);
  lev.zero(c.stream);
  int* h_changed = nullptr;
  PNP_CUDA(cudaMallocHost(&h_changed, sizeof(int)));
  const int g = grid_for(n, 256);
  for (int pass = 0;; pass++) {
    changed.zero(c.stream);
    for (int rep = 0; rep < 8; rep++) { // a few relaxations per host round trip
      if (F == 1) k_level_relax<1><<<g, 256, 0, c.stream>>>(S, lev.p, full, changed.p);
      else k_level_relax<3><<<g, 256, 0, c.stream>>>(S, lev.p, full, changed.p);
      PNP_CHECK_LAUNCH(); c.launches++;
    }
    PNP_CUDA(cudaMemcpyAsync(h_changed, changed.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    if (!*h_changed) break;
    PNP_REQUIRE(pass < (1 << 22), PNP_E_MESH, "level relaxation did not terminate");
  }
  cudaFreeHost(h_changed);
  // number of levels
  DBuf<int> d_max(1);
  size_t bytes = 0;
  cub::DeviceReduce::Max(nullptr, bytes, lev.p, d_max.p, n, c.stream);
  DBuf<char> tmp(bytes);
  PNP_CUDA(cub::DeviceReduce::Max(tmp.p, bytes, lev.p, d_max.p, n, c.stream));
  int maxlev = 0;
  d_max.download(&maxlev, 1, c.stream);
  P->nlev = maxlev + 1;
  int bits = 1; while ((1 << bits) <= maxlev) bits++;
  // sort dofs by level
  DBuf<int> ids(n), slev(n);
  P->dofs.alloc(n);
  k_iota_int<<<g, 256, 0, c.stream>>>(ids.p, n);
  PNP_CHECK_LAUNCH();
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, lev.p, slev.p, ids.p, P->dofs.p, n, 0, bits, c.stream);
  tmp.alloc(bytes);
  PNP_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, bytes, lev.p, slev.p, ids.p, P->dofs.p, n, 0, bits, c.stream));
  P->d_lptr.alloc(P->nlev + 1);
  k_level_starts<<<g, 256, 0, c.stream>>>(slev.p, n, P->nlev, P->d_lptr.p);
  PNP_CHECK_LAUNCH(); c.launches += 4;
  P->lptr = P->d_lptr.to_host(c.stream);
  // segments: runs of small levels share one single-block launch
  for (int l = 0; l < P->nlev;) {
    if (P->lptr[l + 1] - P->lptr[l] > SB_MAX_LEVEL) { P->seg.push_back({l, l + 1, false}); l++; continue; }
    int e = l;
    while (e < P->nlev && P->lptr[e + 1] - P->lptr[e] <= SB_MAX_LEVEL) e++;
    P->seg.push_back({l, e, true});
    l = e;
  }
  return P;
}

std::shared_ptr<SweepPlan> build_plan(Ctx& c, int F, bool full) { return build_plan_view(c, view_of(c), F, full); }

template <int F, int FN> void run_sweep(Ctx& c, const SweepPlan& P, const SweepArgs& a, int dir) {
  const int ns = (int)P.seg.size();
  for (int k = 0; k < ns; k++) {
    const SweepSegment& sg = P.seg[dir > 0 ? k : ns - 1 - k];
    if (sg.single_block) {
      k_sweep_levels<F, FN><<<1, SB_THREADS, 0, c.stream>>>(a, P.dofs.p, P.d_lptr.p, sg.l0, sg.l1, dir);
    } else {
      const int b = P.lptr[sg.l0], e = P.lptr[sg.l0 + 1];
      k_sweep_level<F, FN><<<grid_for(e - b, 256), 256, 0, c.stream>>>(a, P.dofs.p, b, e);
    }
    PNP_CHECK_LAUNCH(); c.launches++;
  }
}
template <int FN> void run_sweep_f(Ctx& c, const SweepPlan& P, const SweepArgs& a, int dir) {
  if (P.F == 1) run_sweep<1, FN>(c, P, a, dir); else run_sweep<3, FN>(c, P, a, dir);
}

SweepPrec& state(Solver& S) {
  if (!S.sweep) S.sweep = std::make_shared<SweepPrec>();
  return *S.sweep;
}

} // namespace

void ssor_setup(Ctx& c, Solver& S, const Matrix& A) {
  PNP_REQUIRE(A.nplanes != PNP_COMPACT_PLANES, PNP_E_ARG, "SSOR sweeps 7-plane PNP matrices only");
  SweepPrec& W = state(S);
  const int F = A.nplanes == 1 ? 1 : 3;
  if (!W.plan_ssor || W.plan_ssor->F != F || W.plan_ssor->n != (long)F * c.n_own) W.plan_ssor = build_plan(c, F, false);
}
// y = SeqSSOR(A, n = prec_steps, w = 1) applied to d, starting from y = 0
void ssor_apply(Ctx& c, Solver& S, const Matrix& A, const double* d, double* y) {
  SweepPrec& W = state(S);
  const SweepPlan& P = *W.plan_ssor;
  vec_zero(c, y, P.n);
  SweepArgs a{view_of(c), A.vals.p, nullptr, c.nslots, d, y};
  for (int s = 0; s < (S.prec_steps > 0 ? S.prec_steps : 1); s++) {
    run_sweep_f<FN_GS>(c, P, a, +1);
    run_sweep_f<FN_GS>(c, P, a, -1);
  }
}

void ilu0_setup(Ctx& c, Solver& S, const Matrix& A) {
  PNP_REQUIRE(A.nplanes != PNP_COMPACT_PLANES, PNP_E_ARG, "ILU0 factors 7-plane PNP matrices only");
  SweepPrec& W = state(S);
  const int F = A.nplanes == 1 ? 1 : 3;
  if (!W.plan_ilu || W.plan_ilu->F != F || W.plan_ilu->n != (long)F * c.n_own) W.plan_ilu = build_plan(c, F, true);
  const size_t need = (size_t)F * F * c.nslots;
  if (W.lu.n != need) W.lu.alloc(need);
  if (F == 1) PNP_CUDA(cudaMemcpyAsync(W.lu.p, A.vals.p, need * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
  else {
    k_planes_7_to_9<<<grid_for(c.nslots, 256), 256, 0, c.stream>>>(A.vals.p, c.nslots, W.lu.p);
    PNP_CHECK_LAUNCH(); c.launches++;
  }
  SweepArgs a{view_of(c), nullptr, W.lu.p, c.nslots, nullptr, nullptr};
  run_sweep_f<FN_ILU_FACTOR>(c, *W.plan_ilu, a, +1);
}
// y = (LU)^-1 d
void ilu0_apply(Ctx& c, Solver& S, const Matrix&, const double* d, double* y) {
  SweepPrec& W = state(S);
  SweepArgs a{view_of(c), nullptr, W.lu.p, c.nslots, d, y};
  run_sweep_f<FN_ILU_FWD>(c, *W.plan_ilu, a, +1);
  run_sweep_f<FN_ILU_BWD>(c, *W.plan_ilu, a, -1);
}

// ---- the same sweeps on any star-layout matrix: the multigrid's Gauss-Seidel smoother (pnp_amg.cu) ----
std::shared_ptr<SweepPlan> sweep_plan_build(Ctx& c, const SweepView& S, int F) { return build_plan_view(c, S, F, false); }
int sweep_plan_levels(const SweepPlan& P) { return P.nlev; }
// one Gauss-Seidel sweep x_i += (d_i - sum_k A_ik x_k) / A_ii over the rows in sweep order (dir > 0) or against it (dir < 0)
void sweep_gs(Ctx& c, const SweepPlan& P, const SweepView& S, const double* vals, long stride, const double* d, double* x, int dir) {
  SweepArgs a{S, vals, nullptr, stride, d, x};
  run_sweep_f<FN_GS>(c, P, a, dir);
}

// number of levels of the sweep schedule (diagnostics / tests); 0 if the solver has none
int sweep_levels(const Solver& S, bool ilu) {
  if (!S.sweep) return 0;
  const auto& p = ilu ? S.sweep->plan_ilu : S.sweep->plan_ssor;
  return p ? p->nlev : 0;
}

} // namespace pnp
