// pnp_star.cuh -- vertex-parallel ("owner computes") assembly over the vertex-star structure.
//
// Data layout (DESIGN.md "HBM layout"): one int32 array `adj` serves both as mesh connectivity and
// as the sparse-matrix column index.  Row v owns slots [rp[v], rp[v+1]):
//   slot rp[v]            : the diagonal (adj = v)
//   slots rp[v]+1 ...     : the neighbours of v in counter-clockwise order (its "ring")
// Bits 27..30 of a ring slot describe the triangle spanned by (v, this neighbour, next neighbour):
//   STAR_HAS_TRI : such a triangle exists (the last slot of a boundary vertex's open fan has none;
//                  the last slot of an interior vertex wraps to the first ring slot)
//   STAR_LI      : element-local index of v in that triangle (so the element's own vertex order,
//                  and with it the reference's quadrature/summation order, can be reconstructed)
//   STAR_CW      : the element is stored clockwise (then next-in-ring is its cyclic successor)
// Vectors are vertex-blocked: dof (v, field k) lives at F*v + k.  Matrix values are stored as
// NPLANES planes of nslots doubles (PNP: 7 planes, see pnp_plane(), or the compact 5, see pnp_block()).
//
// This replaces PDELab's element loop + scatter (GridOperator::residual/jacobian, SURVEY App. A.2;
// call sites /root/reference/src/stationary_pnp.hh:240-246): every residual entry / matrix slot is
// written exactly once by exactly one thread -- no atomics, no zero-fill, deterministic.
#pragma once
#include "pnp_elem.cuh"
#include "pnp_setup_algos.cuh"

namespace pnp {


struct XY { double x, y; };

struct StarView {
  const int* rp;              // nv+1
  const unsigned* adj;        // nslots
  const XY* xy;               // nv (internal numbering)
  const unsigned char* dmask; // nv: bit c = vertex is Dirichlet for BC component c
  int nv;
};

template <int OP> struct VData {
  static constexpr int F = OpTraits<OP>::F;
  static constexpr int NA = OpTraits<OP>::NAUX > 0 ? OpTraits<OP>::NAUX : 1;
  double x, y, u[F], a[NA];
};

template <int OP>
PNP_HD VData<OP> load_vertex(const StarView& M, const double* u, const double* aux0, const double* aux1, int w) {
  VData<OP> d;
  const XY p = M.xy[w];
  d.x = p.x; d.y = p.y;
#pragma unroll
  for (int k = 0; k < VData<OP>::F; k++) d.u[k] = u ? u[(long)VData<OP>::F * w + k] : 0.0;
  d.a[0] = 0.0;
  if (OpTraits<OP>::NAUX >= 1) d.a[0] = aux0[w];
  if (OpTraits<OP>::NAUX >= 2) d.a[1] = aux1[w];
  return d;
}

// gathers element-local arrays from the three vertices given in ELEMENT-LOCAL order
template <int OP>
PNP_HD Geo gather_local(const VData<OP>& A0, const VData<OP>& A1, const VData<OP>& A2,
                        double (*xl)[3], double (*aux)[3]) {
#pragma unroll
  for (int k = 0; k < VData<OP>::F; k++) { xl[k][0] = A0.u[k]; xl[k][1] = A1.u[k]; xl[k][2] = A2.u[k]; }
#pragma unroll
  for (int a = 0; a < VData<OP>::NA; a++) { aux[a][0] = A0.a[a]; aux[a][1] = A1.a[a]; aux[a][2] = A2.a[a]; }
  return make_geo(A0.x, A0.y, A1.x, A1.y, A2.x, A2.y);
}

template <int OP, int I>
PNP_HD void tri_rows(const VData<OP>& A0, const VData<OP>& A1, const VData<OP>& A2, const PhysParams& P, double* out) {
  double xl[VData<OP>::F][3], aux[VData<OP>::NA][3];
  const Geo G = gather_local<OP>(A0, A1, A2, xl, aux);
  rows_faithful<OP, I>(G, P, xl, aux, out);
}

// decode: which ring neighbour is the cyclic successor (n) / predecessor (p) of v in the element
//   element-local order: a[li] = v, a[(li+1)%3] = n, a[(li+2)%3] = p
template <int OP>
PNP_HD void residual_tri(unsigned flags, const VData<OP>& V, const VData<OP>& cur, const VData<OP>& nxt,
                         const PhysParams& P, double* out) {
  const int li = (flags >> STAR_LI_SHIFT) & 3;
  const bool cw = flags & STAR_CW;
  const VData<OP>& N = cw ? nxt : cur;
  const VData<OP>& Pp = cw ? cur : nxt;
  if (li == 0) tri_rows<OP, 0>(V, N, Pp, P, out);
  else if (li == 1) tri_rows<OP, 1>(Pp, V, N, P, out);
  else tri_rows<OP, 2>(N, Pp, V, P, out);
}

// Volume part of residual row(s) of vertex v: out[k] = sum over incident elements (ring order).
template <int OP, bool FAITHFUL = false>
PNP_HD void residual_row(const StarView& M, const PhysParams& P, const double* u, const double* aux0,
                         const double* aux1, int v, double* out) {
  constexpr int F = OpTraits<OP>::F;
#pragma unroll
  for (int k = 0; k < F; k++) out[k] = 0.0;
  const int s0 = M.rp[v] + 1, s1 = M.rp[v + 1];
  if (s0 >= s1) return;
  const VData<OP> V = load_vertex<OP>(M, u, aux0, aux1, v);
  unsigned a_cur = M.adj[s0];
  const unsigned a_first = a_cur;
  VData<OP> cur = load_vertex<OP>(M, u, aux0, aux1, (int)(a_cur & STAR_VMASK));
  const VData<OP> first = cur;
  for (int s = s0; s < s1; s++) {
    const bool last = (s + 1 == s1);
    unsigned a_nxt = last ? a_first : M.adj[s + 1];
    VData<OP> nxt;
    if (last) nxt = first; else nxt = load_vertex<OP>(M, u, aux0, aux1, (int)(a_nxt & STAR_VMASK));
    if (a_cur & STAR_HAS_TRI) {
      double rl[F];
#pragma unroll
      for (int k = 0; k < F; k++) rl[k] = 0.0;
      // FAITHFUL: the element's own vertex order (the reference's operation order, needed by the FD Jacobian);
      // otherwise the triangle is taken as (v, this neighbour, next neighbour): same integrals (the quadrature rules
      // are symmetric), no branch on the element-local index, results equal up to rounding
      if (FAITHFUL) residual_tri<OP>(a_cur, V, cur, nxt, P, rl);
      else tri_rows<OP, 0>(V, cur, nxt, P, rl);
#pragma unroll
      for (int k = 0; k < F; k++) out[k] += rl[k];
    }
    a_cur = a_nxt; cur = nxt;
  }
}

// ---- Jacobian ------------------------------------------------------------------------------
enum : int { JAC_FD_FAITHFUL = 0, JAC_ANALYTIC = 1 };

template <int OP, int I, int MODE, int NP>
PNP_HD void tri_jac(const VData<OP>& A0, const VData<OP>& A1, const VData<OP>& A2, const PhysParams& P, double eps,
                    double (*blk)[NP]) {
  double xl[VData<OP>::F][3], aux[VData<OP>::NA][3];
  const Geo G = gather_local<OP>(A0, A1, A2, xl, aux);
  if constexpr (NP != OpTraits<OP>::NPLANES) {
    static_assert(OP == OP_PNP && NP == PNP_COMPACT_PLANES && MODE == JAC_ANALYTIC, "compact layout: exact PNP Jacobian only");
    jac_rows_exact_compact<I>(G, P, xl, blk);
  } else if (MODE == JAC_FD_FAITHFUL) jac_rows_fd<OP, I>(G, P, xl, aux, eps, blk);
  else jac_rows_exact<OP, I>(G, P, xl, aux, blk);
}

// Dirichlet treatment of one block (SURVEY App. A.2): entries whose row or column dof is
// constrained are dropped; a constrained row keeps a unit diagonal.  rb/cb = Dirichlet bits of the
// row/column vertex restricted to this operator's fields.  The compact layout's vertices are constrained in all three
// fields or in none (pnp_jacobian_planes): the block goes as a whole, a constrained row keeps L = 1, D = 0.
template <int OP, int NP = OpTraits<OP>::NPLANES>
PNP_HD void mask_block(double* b, unsigned rb, unsigned cb, bool diagonal) {
  if (NP == PNP_COMPACT_PLANES) {
    if ((rb | cb) & 7u) {
#pragma unroll
      for (int p = 0; p < NP; p++) b[p] = 0.0;
      if (diagonal && (rb & 1u)) b[0] = 1.0;
    }
  } else if (OP == OP_PNP) {
#pragma unroll
    for (int ki = 0; ki < 3; ki++)
#pragma unroll
      for (int kj = 0; kj < 3; kj++) {
        const int pl = pnp_plane(ki, kj);
        if (pl < 0) continue;
        if (((rb >> ki) & 1u) | ((cb >> kj) & 1u)) b[pl] = (diagonal && ki == kj && ((rb >> ki) & 1u)) ? 1.0 : 0.0;
      }
  } else {
    if ((rb | cb) & 1u) b[0] = (diagonal && (rb & 1u)) ? 1.0 : 0.0;
  }
}

// Dirichlet bits of vertex w for this operator: PNP uses components 0,1,2 as fields; scalar
// operators use the single component `comp0` their BCType was built with (btype.hh:21-53).
template <int OP> PNP_HD unsigned dir_bits(const StarView& M, int w, int comp0) {
  const unsigned m = M.dmask[w];
  return OP == OP_PNP ? (m & 7u) : ((m >> comp0) & 1u);
}

// Assembles the block row of vertex v into vals[plane*stride + slot - sbase] (sbase != 0: `vals` is a staging tile
// that starts at global slot sbase), in the operator's NPLANES planes or, NP = PNP_COMPACT_PLANES, the compact layout.
template <int OP, int MODE, int NP = OpTraits<OP>::NPLANES>
PNP_HD void jacobian_row(const StarView& M, const PhysParams& P, const double* u, const double* aux0,
                         const double* aux1, double eps, int comp0, int v, double* vals, long stride, int sbase = 0) {
  vals -= sbase; // only entries [sbase, ...) of a plane are touched
  const int sd = M.rp[v], s0 = sd + 1, s1 = M.rp[v + 1];
  const unsigned rb = dir_bits<OP>(M, v, comp0);
  double diag[NP], carry[NP];
#pragma unroll
  for (int p = 0; p < NP; p++) { diag[p] = 0.0; carry[p] = 0.0; }
  bool closed = false;
  unsigned cb_first = 0;
  if (s0 < s1) {
    const VData<OP> V = load_vertex<OP>(M, u, aux0, aux1, v);
    unsigned a_cur = M.adj[s0];
    const unsigned a_first = a_cur;
    VData<OP> cur = load_vertex<OP>(M, u, aux0, aux1, (int)(a_cur & STAR_VMASK));
    const VData<OP> first = cur;
    unsigned cb_cur = dir_bits<OP>(M, (int)(a_cur & STAR_VMASK), comp0);
    cb_first = cb_cur;
    for (int s = s0; s < s1; s++) {
      const bool last = (s + 1 == s1);
      const unsigned a_nxt = last ? a_first : M.adj[s + 1];
      VData<OP> nxt;
      if (last) nxt = first; else nxt = load_vertex<OP>(M, u, aux0, aux1, (int)(a_nxt & STAR_VMASK));
      double val[NP];
#pragma unroll
      for (int p = 0; p < NP; p++) val[p] = carry[p];
      if (a_cur & STAR_HAS_TRI) {
        // blk[jl]: contributions to the columns of element-local vertex jl
        double blk[3][NP];
#pragma unroll
        for (int j = 0; j < 3; j++)
#pragma unroll
          for (int p = 0; p < NP; p++) blk[j][p] = 0.0;
        const double *bv, *bcur, *bnxt;
        if (MODE == JAC_ANALYTIC) { // vertex-centric order (v, this neighbour, next neighbour): no branch on li
          tri_jac<OP, 0, MODE, NP>(V, cur, nxt, P, eps, blk);
          bv = blk[0]; bcur = blk[1]; bnxt = blk[2];
        } else {
          const int li = (a_cur >> STAR_LI_SHIFT) & 3;
          const bool cw = a_cur & STAR_CW;
          const VData<OP>& N = cw ? nxt : cur;
          const VData<OP>& Pp = cw ? cur : nxt;
          // local column index of: v -> li, n -> (li+1)%3, p -> (li+2)%3
          const double *bn, *bp;
          if (li == 0) { tri_jac<OP, 0, MODE, NP>(V, N, Pp, P, eps, blk); bv = blk[0]; bn = blk[1]; bp = blk[2]; }
          else if (li == 1) { tri_jac<OP, 1, MODE, NP>(Pp, V, N, P, eps, blk); bv = blk[1]; bn = blk[2]; bp = blk[0]; }
          else { tri_jac<OP, 2, MODE, NP>(N, Pp, V, P, eps, blk); bv = blk[2]; bn = blk[0]; bp = blk[1]; }
          bcur = cw ? bp : bn;
          bnxt = cw ? bn : bp;
        }
#pragma unroll
        for (int p = 0; p < NP; p++) { diag[p] += bv[p]; val[p] += bcur[p]; carry[p] = bnxt[p]; }
        closed = last;
      } else {
#pragma unroll
        for (int p = 0; p < NP; p++) carry[p] = 0.0;
      }
      if (!(last && closed && s == s0)) { // (a one-slot closed ring cannot exist)
        mask_block<OP, NP>(val, rb, cb_cur, false);
#pragma unroll
        for (int p = 0; p < NP; p++) vals[p * stride + s] = val[p];
      }
      a_cur = a_nxt; cur = nxt;
      cb_cur = last ? cb_first : dir_bits<OP>(M, (int)(a_nxt & STAR_VMASK), comp0);
    }
    if (closed) { // the wrap-around triangle's contribution to the first ring slot
      mask_block<OP, NP>(carry, rb, cb_first, false);
#pragma unroll
      for (int p = 0; p < NP; p++) vals[p * stride + s0] += carry[p];
    }
  }
  mask_block<OP, NP>(diag, rb, rb, true);
#pragma unroll
  for (int p = 0; p < NP; p++) vals[p * stride + sd] = diag[p];
}

// Value planes of a PNP Jacobian that only the star SpMV and diagonal-block consumers read (solver_ok: no SSOR / ILU0 /
// Gauss-Seidel sweeps): the compact layout for the exact derivative on linear elements when every surface of the
// parameter set has its three components all Dirichlet or all not (btype: 3 per surface, 0 = Dirichlet); else 7.
// Decided from the parameters alone, so every rank of a partitioned mesh takes the same layout.
inline int pnp_jacobian_planes(int mode, int degree, bool solver_ok, const int* btype, int n_surfaces) {
  if (mode != JAC_ANALYTIC || degree != 1 || !solver_ok) return OpTraits<OP_PNP>::NPLANES;
  for (int s = 0; s < n_surfaces; s++) {
    const bool d0 = btype[3 * s] == 0;
    if ((btype[3 * s + 1] == 0) != d0 || (btype[3 * s + 2] == 0) != d0) return OpTraits<OP_PNP>::NPLANES;
  }
  return PNP_COMPACT_PLANES;
}

// ---- boundary term (alpha_boundary) -------------------------------------------------------------
// Sum of the boundary-face contributions to one vertex, faces in ascending face order
// (deterministic).  items[] = face*4 + role (element-local index of the vertex in that face's
// element).  Field k uses BC component (F==3 ? k : comp0) for the "not Dirichlet" test of the face
// and for the flux (pnp_operator.hh:252-313, pb_operator.hh:137-190).
PNP_HD void boundary_vertex_sum(const StarView& M, const PhysParams& P, const BFace* faces, const int* items, int i0,
                                int i1, const double* surf_flux, const unsigned char* surf_dir, int F, int comp0,
                                double* acc) {
  acc[0] = acc[1] = acc[2] = 0.0;
  for (int it = i0; it < i1; it++) {
    const BFace b = faces[items[it] >> 2];
    const int role = items[it] & 3;
    const XY A = M.xy[b.v[face_v(b.f, 0)]], B = M.xy[b.v[face_v(b.f, 1)]];
    for (int k = 0; k < F; k++) {
      const int comp = F == 3 ? k : comp0;
      if ((surf_dir[b.phys] >> comp) & 1) continue; // isDirichlet(ig, x) -> no flux term
      double out[3] = {0.0, 0.0, 0.0};
      boundary_face(b.f, A.x, A.y, B.x, B.y, surf_flux[3 * b.phys + comp], P, out);
      acc[k] += out[role];
    }
  }
}

} // namespace pnp
