// pnp_elem.cuh -- element-level fp64 math of the five local operators (P1 triangles).
//
// Everything here is a __host__ __device__ function of plain scalars so that the CUDA kernels
// (pnp_assembly.cu) and the CPU logic harness under tests/host_harness/ compile the same source.
// The harness is test infrastructure; the product library only instantiates the device side.
//
// "Faithful" functions reproduce, operation by operation, what the reference's alpha_volume does
// for ONE local test function i (the rows of an element residual are independent, so a
// vertex-parallel gather can evaluate just its own row and still get the reference's bits):
//   PnpOperator::alpha_volume        /root/reference/src/pnp_operator.hh:98-194
//   PBOperator::alpha_volume         pb_operator.hh:74-120
//   PoissonOperator::alpha_volume    poisson_operator.hh:74-126
//   DiffusionOperator::alpha_volume  diffusion_operator.hh:64-111
//   DiffusionTOperator::alpha_volume diffusion_toperator.hh:58-72
// and NumericalJacobianVolume (SURVEY App. A.3) on top of them.  They must be compiled without
// FMA contraction (nvcc -fmad=false / g++ -ffp-contract=off).
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define PNP_HD __host__ __device__ __forceinline__
#else
#define PNP_HD inline
#endif

namespace pnp {

enum : int { OP_PB = 0, OP_POISSON = 1, OP_DIFFUSION = 2, OP_MASS = 3, OP_PNP = 4 };

// physical parameters the element integrals need (Sysparams subset, sysparams.hh:10-37)
struct PhysParams {
  double PI;     // 3.1415 in the reference (pnp_operator.hh:20)
  double l_b, c0;
  double valency; // DiffusionOperator ctor argument (instationary_pnp_from_pb_md.hh:358,360)
  int cylindrical;
};

template <int OP> struct OpTraits;
template <> struct OpTraits<OP_PB>        { static constexpr int F = 1, NQ = 4, NAUX = 0, NPLANES = 1; };
template <> struct OpTraits<OP_POISSON>   { static constexpr int F = 1, NQ = 4, NAUX = 2, NPLANES = 1; };
template <> struct OpTraits<OP_DIFFUSION> { static constexpr int F = 1, NQ = 3, NAUX = 1, NPLANES = 1; };
template <> struct OpTraits<OP_MASS>      { static constexpr int F = 1, NQ = 7, NAUX = 0, NPLANES = 1; };
// PNP: 7 structurally non-zero 3x3-block entries (phi,phi)(phi,+)(phi,-)(+,phi)(+,+)(-,phi)(-,-);
// the (+,-) and (-,+) couplings are exact zeros, also under the reference's finite differences.
template <> struct OpTraits<OP_PNP>       { static constexpr int F = 3, NQ = 4, NAUX = 0, NPLANES = 7; };

// plane index of block entry (row field ki, column field kj) for the PNP system, -1 if structurally zero
PNP_HD constexpr int pnp_plane(int ki, int kj) {
  return ki == 0 ? kj : (ki == 1 ? (kj == 0 ? 3 : (kj == 1 ? 4 : -1)) : (kj == 0 ? 5 : (kj == 2 ? 6 : -1)));
}

// The exact-derivative PNP Jacobian also comes in a compact layout of 5 planes: the residual has unit coefficients on
// grad(phi).grad(v), grad(c+).grad(v) and grad(c-).grad(v), so the three diagonal blocks share one Laplacian L, and
// (phi,c-) is the negation of (phi,c+):
//   plane 0: L = (phi,phi)    1: M = (phi,c+) = -(phi,c-)    2: (c+,phi)    3: (c-,phi)
//   plane 4: D, the drift:   (c+,c+) = L - D,  (c-,c-) = L + D
// It needs every constrained vertex to be constrained in all three fields (one unit diagonal L = 1, D = 0 per vertex).
// A star SpMV then reads 44 B per slot instead of 60.
constexpr int PNP_COMPACT_PLANES = 5;

// the 3x3 block [a b c; d e 0; f 0 g] of one slot from its NP value planes (1: scalar a; 5: compact; 7: pnp_plane())
struct PnpBlock {
  double a, b, c, d, e, f, g;
  PNP_HD double at(int ki, int kj) const {
    return ki == 0 ? (kj == 0 ? a : (kj == 1 ? b : c)) : (ki == 1 ? (kj == 0 ? d : (kj == 1 ? e : 0.0)) : (kj == 0 ? f : (kj == 2 ? g : 0.0)));
  }
};
template <int NP> PNP_HD PnpBlock pnp_block(const double* v) {
  static_assert(NP == 1 || NP == 5 || NP == 7, "PNP value planes: 1, 5 or 7");
  if (NP == 1) return PnpBlock{v[0], 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (NP == 5) return PnpBlock{v[0], v[1], -v[1], v[2], v[0] - v[4 % NP], v[3 % NP], v[0] + v[4 % NP]};
  return PnpBlock{v[0], v[1 % NP], v[2 % NP], v[3 % NP], v[4 % NP], v[5 % NP], v[6 % NP]};
}
// ... of slot s of NP planes `stride` doubles apart
template <int NP> PNP_HD PnpBlock pnp_block_at(const double* vals, long stride, long s) {
  double v[NP];
#pragma unroll
  for (int p = 0; p < NP; p++) v[p] = vals[p * stride + s];
  return pnp_block<NP>(v);
}

// Quadrature tables (dune-geometry simplex rules; SURVEY App. A.6): point q of the NQ-point rule.
template <int NQ> PNP_HD void quad_point(int q, double& xi0, double& xi1, double& w);
template <> PNP_HD void quad_point<3>(int q, double& xi0, double& xi1, double& w) {
  w = 0.5 / 3.0;
  xi0 = q == 0 ? 4.0 / 6.0 : 1.0 / 6.0;
  xi1 = q == 1 ? 4.0 / 6.0 : 1.0 / 6.0;
}
template <> PNP_HD void quad_point<4>(int q, double& xi0, double& xi1, double& w) {
  w = q == 0 ? 0.5 * (-27.0 / 48.0) : 0.5 * (25.0 / 48.0);
  xi0 = q == 0 ? 10.0 / 30.0 : (q == 1 ? 18.0 / 30.0 : 6.0 / 30.0);
  xi1 = q == 0 ? 10.0 / 30.0 : (q == 2 ? 18.0 / 30.0 : 6.0 / 30.0);
}
template <> PNP_HD void quad_point<7>(int q, double& xi0, double& xi1, double& w) {
  const double a = 0.79742698535308732240, b = 0.10128650732345633880;
  const double c = 0.05971587178976982045, d = 0.47014206410511508977;
  const double wb = 0.5 * 0.12593918054482715260, wd = 0.5 * 0.13239415278850618074;
  if (q == 0) { xi0 = 1.0 / 3.0; xi1 = 1.0 / 3.0; w = 0.5 * 0.225; }
  else if (q < 4) { w = wb; xi0 = q == 1 ? a : b; xi1 = q == 2 ? a : b; }
  else { w = wd; xi0 = q == 4 ? c : d; xi1 = q == 5 ? c : d; }
}

// sinh for the Poisson-Boltzmann source term (pb_operator.hh:117), built from +, -, *, / and floor only, so that the device
// (compiled -fmad=false) and the CPU oracle (-ffp-contract=off), which carries the same sequence of operations, get the same
// BITS: NumericalJacobianVolume divides differences of the residual by delta ~ 1e-11, and a last-bit difference between
// two libm's sinh would show up ten thousand times larger in the FD Jacobian (SURVEY H1).  |error| <= 4 ulp for |x| < 700.
PNP_HD double pnp_pow2(int k) { // 2^k, -1022 <= k <= 1023
  const unsigned long long bits = (unsigned long long)(k + 1023) << 52;
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)bits);
#else
  double d; __builtin_memcpy(&d, &bits, sizeof d); return d;
#endif
}
PNP_HD double pnp_sinh(double x) {
  const double a = x < 0.0 ? -x : x;
  double r;
  if (a < 0.35) { // odd Taylor series, Horner in x^2 (next term x^17/17! < 1e-22)
    const double t = a * a;
    double p = 1.0 / 1307674368000.0;        // 1/15!
    p = p * t + 1.0 / 6227020800.0;          // 1/13!
    p = p * t + 1.0 / 39916800.0;            // 1/11!
    p = p * t + 1.0 / 362880.0;              // 1/9!
    p = p * t + 1.0 / 5040.0;                // 1/7!
    p = p * t + 1.0 / 120.0;                 // 1/5!
    p = p * t + 1.0 / 6.0;                   // 1/3!
    r = a + a * (t * p);
  } else {        // (e^a - e^-a) / 2 with e^a = 2^k e^s, |s| <= ln2 / 2
    const double kf = floor(a * 1.44269504088896338700e+00 + 0.5);
    const double s = (a - kf * 6.93147180369123816490e-01) - kf * 1.90821492927058770002e-10;
    double p = 1.0 / 87178291200.0;          // 1/14!
    p = p * s + 1.0 / 6227020800.0;
    p = p * s + 1.0 / 479001600.0;
    p = p * s + 1.0 / 39916800.0;
    p = p * s + 1.0 / 3628800.0;
    p = p * s + 1.0 / 362880.0;
    p = p * s + 1.0 / 40320.0;
    p = p * s + 1.0 / 5040.0;
    p = p * s + 1.0 / 720.0;
    p = p * s + 1.0 / 120.0;
    p = p * s + 1.0 / 24.0;
    p = p * s + 1.0 / 6.0;
    p = p * s + 0.5;
    p = p * s + 1.0;
    p = p * s + 1.0;
    const int k = (int)kf;
    const double e = p * pnp_pow2(k / 2) * pnp_pow2(k - k / 2);
    r = 0.5 * e - 0.5 / e;
  }
  return x < 0.0 ? -r : r;
}

// Affine geometry of one triangle with vertices in ELEMENT-LOCAL order.
struct Geo {
  double y0, y1, y2;   // for geometry().global()[1]
  double g[3][2];      // J^{-T} * reference gradient of local basis i
  double detabs;       // integrationElement
};
PNP_HD Geo make_geo(double x0, double y0, double x1, double y1, double x2, double y2) {
  Geo G;
  G.y0 = y0; G.y1 = y1; G.y2 = y2;
  const double j00 = x1 - x0, j01 = x2 - x0, j10 = y1 - y0, j11 = y2 - y0;
  const double det = j00 * j11 - j01 * j10;
  const double di = 1.0 / det;
  const double t00 = j11 * di, t01 = -j10 * di, t10 = -j01 * di, t11 = j00 * di; // J^{-T}
  G.detabs = fabs(det);
  // FieldMatrix::mv with reference gradients (-1,-1),(1,0),(0,1): y = 0; y += a*x0; y += b*x1
  G.g[0][0] = (0.0 + t00 * -1.0) + t01 * -1.0;  G.g[0][1] = (0.0 + t10 * -1.0) + t11 * -1.0;
  G.g[1][0] = (0.0 + t00 * 1.0) + t01 * 0.0;    G.g[1][1] = (0.0 + t10 * 1.0) + t11 * 0.0;
  G.g[2][0] = (0.0 + t00 * 0.0) + t01 * 1.0;    G.g[2][1] = (0.0 + t10 * 0.0) + t11 * 1.0;
  return G;
}
PNP_HD double dot2(const double* a, const double* b) { // FieldVector::operator*
  double r = 0.0; r += a[0] * b[0]; r += a[1] * b[1]; return r;
}

// ---------------------------------------------------------------------------------------------
// Faithful residual rows.  xl[k][i] = local coefficient of field k at element-local vertex i,
// aux[a][i] = coefficient field a (Poisson: c+, c-; diffusion: Phi) at local vertex i.
// ACCUMULATES the contribution of this element to test function I of every field into out[k].
// ---------------------------------------------------------------------------------------------
// (I may be a run-time value: it only selects one basis value and one gradient; rows_faithful<OP, I> below fixes it at
// compile time.  Same operations in the same order either way.)
template <int OP>
PNP_HD void rows_faithful_at(const Geo& G, const PhysParams& P, const double (*xl)[3], const double (*aux)[3], const int I,
                             double* out) {
  constexpr int NQ = OpTraits<OP>::NQ;
  const double PI = P.PI;
  const double gI[2] = {I == 0 ? G.g[0][0] : (I == 1 ? G.g[1][0] : G.g[2][0]), I == 0 ? G.g[0][1] : (I == 1 ? G.g[1][1] : G.g[2][1])};
#pragma unroll
  for (int q = 0; q < NQ; q++) {
    double xi0, xi1, w;
    quad_point<NQ>(q, xi0, xi1, w);
    const double phi[3] = {1.0 - xi0 - xi1, xi0, xi1};
    const double phiI = I == 0 ? phi[0] : (I == 1 ? phi[1] : phi[2]);
    const double gy = G.y0 + (G.y1 - G.y0) * xi0 + (G.y2 - G.y0) * xi1;
    double factor = w * G.detabs;
    if (OP == OP_PNP) {
      if (P.cylindrical) factor *= gy * 2 * PI;
      double u[3], gu[3][2];
#pragma unroll
      for (int k = 0; k < 3; k++) {
        u[k] = 0.0;
#pragma unroll
        for (int i = 0; i < 3; i++) u[k] += xl[k][i] * phi[i];
        gu[k][0] = 0.0; gu[k][1] = 0.0;
#pragma unroll
        for (int i = 0; i < 3; i++) { gu[k][0] += xl[k][i] * G.g[i][0]; gu[k][1] += xl[k][i] * G.g[i][1]; }
      }
      out[0] += (dot2(gu[0], gI) + 4 * PI * P.l_b * (u[1] - u[2]) * phiI) * factor;
      out[1] += (dot2(gu[1], gI) - u[1] * dot2(gu[0], gI)) * factor;
      out[2] += (dot2(gu[2], gI) + u[2] * dot2(gu[0], gI)) * factor;
    } else if (OP == OP_PB || OP == OP_POISSON) {
      if (P.cylindrical) factor *= gy * 2 * PI;
      double u = 0.0, gu[2] = {0.0, 0.0};
#pragma unroll
      for (int i = 0; i < 3; i++) u += xl[0][i] * phi[i];
#pragma unroll
      for (int i = 0; i < 3; i++) { gu[0] += xl[0][i] * G.g[i][0]; gu[1] += xl[0][i] * G.g[i][1]; }
      double src;
      if (OP == OP_PB) src = 8 * PI * P.l_b * P.c0 * pnp_sinh(u);
      else {
        double cp = 0.0, cm = 0.0;
#pragma unroll
        for (int i = 0; i < 3; i++) cp += aux[0][i] * phi[i];
#pragma unroll
        for (int i = 0; i < 3; i++) cm += aux[1][i] * phi[i];
        src = 1 * P.l_b * 4 * PI * (cm - cp);
      }
      out[0] += (dot2(gu, gI) + src * phiI) * factor;
    } else if (OP == OP_DIFFUSION) {
      double u = 0.0, gu[2] = {0.0, 0.0}, gP[2] = {0.0, 0.0};
#pragma unroll
      for (int i = 0; i < 3; i++) u += xl[0][i] * phi[i];
#pragma unroll
      for (int i = 0; i < 3; i++) { gu[0] += xl[0][i] * G.g[i][0]; gu[1] += xl[0][i] * G.g[i][1]; }
#pragma unroll
      for (int i = 0; i < 3; i++) { gP[0] += aux[0][i] * G.g[i][0]; gP[1] += aux[0][i] * G.g[i][1]; }
      const double a = 0;
      out[0] += (dot2(gu, gI) + u * P.valency * dot2(gP, gI) + a * u * phiI) * factor;
    } else { // OP_MASS
      double u = 0.0;
#pragma unroll
      for (int i = 0; i < 3; i++) u += xl[0][i] * phi[i];
      out[0] += u * phiI * factor;
    }
  }
}
template <int OP, int I>
PNP_HD void rows_faithful(const Geo& G, const PhysParams& P, const double (*xl)[3], const double (*aux)[3], double* out) {
  rows_faithful_at<OP>(G, P, xl, aux, I, out);
}

// ---------------------------------------------------------------------------------------------
// Row I of the element Jacobian, as NPLANES values per column vertex: blk[jl][plane].
// FD-faithful: NumericalJacobianVolume restricted to row I (forward difference, delta =
// eps*(1+|u_j|), column order = child-major local DOFs).  ACCUMULATES into blk.
// ---------------------------------------------------------------------------------------------
template <int OP, int I>
PNP_HD void jac_rows_fd(const Geo& G, const PhysParams& P, double (*xl)[3], const double (*aux)[3], double eps,
                        double (*blk)[OpTraits<OP>::NPLANES]) {
  constexpr int F = OpTraits<OP>::F;
  double down[F];
#pragma unroll
  for (int k = 0; k < F; k++) down[k] = 0.0;
  rows_faithful<OP, I>(G, P, xl, aux, down);
#pragma unroll
  for (int kj = 0; kj < F; kj++)
#pragma unroll
    for (int jl = 0; jl < 3; jl++) {
      const double keep = xl[kj][jl];
      const double delta = eps * (1.0 + fabs(keep));
      xl[kj][jl] = keep + delta;
      double up[F];
#pragma unroll
      for (int k = 0; k < F; k++) up[k] = 0.0;
      rows_faithful<OP, I>(G, P, xl, aux, up);
      xl[kj][jl] = keep;
      if (OP == OP_PNP) {
#pragma unroll
        for (int ki = 0; ki < 3; ki++) {
          const int pl = pnp_plane(ki, kj);
          if (pl >= 0) blk[jl][pl] += (up[ki] - down[ki]) / delta;
        }
      } else {
        blk[jl][0] += (up[0] - down[0]) / delta;
      }
    }
}

// Exact derivative of the same residual rows (fast path; not in the reference, which only has FD).
template <int OP, int I>
PNP_HD void jac_rows_exact(const Geo& G, const PhysParams& P, const double (*xl)[3], const double (*aux)[3],
                           double (*blk)[OpTraits<OP>::NPLANES]) {
  constexpr int NQ = OpTraits<OP>::NQ;
  double K[3]; // grad phi_j . grad phi_I
#pragma unroll
  for (int j = 0; j < 3; j++) K[j] = G.g[j][0] * G.g[I][0] + G.g[j][1] * G.g[I][1];
  double gP[2] = {0.0, 0.0}; // gradient of the potential (PNP: field 0; diffusion: aux 0)
  if (OP == OP_PNP) {
#pragma unroll
    for (int i = 0; i < 3; i++) { gP[0] += xl[0][i] * G.g[i][0]; gP[1] += xl[0][i] * G.g[i][1]; }
  } else if (OP == OP_DIFFUSION) {
#pragma unroll
    for (int i = 0; i < 3; i++) { gP[0] += aux[0][i] * G.g[i][0]; gP[1] += aux[0][i] * G.g[i][1]; }
  }
  const double dPI = gP[0] * G.g[I][0] + gP[1] * G.g[I][1];
#pragma unroll
  for (int q = 0; q < NQ; q++) {
    double xi0, xi1, w;
    quad_point<NQ>(q, xi0, xi1, w);
    const double phi[3] = {1.0 - xi0 - xi1, xi0, xi1};
    double factor = w * G.detabs;
    if ((OP == OP_PNP || OP == OP_PB || OP == OP_POISSON) && P.cylindrical) {
      const double gy = G.y0 + (G.y1 - G.y0) * xi0 + (G.y2 - G.y0) * xi1;
      factor *= gy * 2 * P.PI;
    }
    if (OP == OP_PNP) {
      double up = 0.0, um = 0.0;
#pragma unroll
      for (int i = 0; i < 3; i++) { up += xl[1][i] * phi[i]; um += xl[2][i] * phi[i]; }
      const double kap = 4 * P.PI * P.l_b;
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const double m = kap * phi[j] * phi[I] * factor;
        blk[j][0] += K[j] * factor;
        blk[j][1] += m;
        blk[j][2] -= m;
        blk[j][3] -= up * K[j] * factor;
        blk[j][4] += (K[j] - phi[j] * dPI) * factor;
        blk[j][5] += um * K[j] * factor;
        blk[j][6] += (K[j] + phi[j] * dPI) * factor;
      }
    } else {
      double u = 0.0;
      if (OP == OP_PB) {
#pragma unroll
        for (int i = 0; i < 3; i++) u += xl[0][i] * phi[i];
      }
      const double ch = OP == OP_PB ? 8 * P.PI * P.l_b * P.c0 * cosh(u) : 0.0;
#pragma unroll
      for (int j = 0; j < 3; j++) {
        double v;
        if (OP == OP_PB) v = K[j] + ch * phi[j] * phi[I];
        else if (OP == OP_POISSON) v = K[j];
        else if (OP == OP_DIFFUSION) v = K[j] + phi[j] * P.valency * dPI;
        else v = phi[j] * phi[I];
        blk[j][0] += v * factor;
      }
    }
  }
}

// The same exact derivative of the PNP rows in the compact layout (PNP_COMPACT_PLANES).  L, M, (c+,phi) and (c-,phi) are
// the operations of jac_rows_exact in the same order; D collects the drift terms that planes 4 and 6 add to K there.
template <int I>
PNP_HD void jac_rows_exact_compact(const Geo& G, const PhysParams& P, const double (*xl)[3],
                                   double (*blk)[PNP_COMPACT_PLANES]) {
  constexpr int NQ = OpTraits<OP_PNP>::NQ;
  double K[3];
#pragma unroll
  for (int j = 0; j < 3; j++) K[j] = G.g[j][0] * G.g[I][0] + G.g[j][1] * G.g[I][1];
  double gP[2] = {0.0, 0.0};
#pragma unroll
  for (int i = 0; i < 3; i++) { gP[0] += xl[0][i] * G.g[i][0]; gP[1] += xl[0][i] * G.g[i][1]; }
  const double dPI = gP[0] * G.g[I][0] + gP[1] * G.g[I][1];
#pragma unroll
  for (int q = 0; q < NQ; q++) {
    double xi0, xi1, w;
    quad_point<NQ>(q, xi0, xi1, w);
    const double phi[3] = {1.0 - xi0 - xi1, xi0, xi1};
    double factor = w * G.detabs;
    if (P.cylindrical) {
      const double gy = G.y0 + (G.y1 - G.y0) * xi0 + (G.y2 - G.y0) * xi1;
      factor *= gy * 2 * P.PI;
    }
    double up = 0.0, um = 0.0;
#pragma unroll
    for (int i = 0; i < 3; i++) { up += xl[1][i] * phi[i]; um += xl[2][i] * phi[i]; }
    const double kap = 4 * P.PI * P.l_b;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const double m = kap * phi[j] * phi[I] * factor;
      blk[j][0] += K[j] * factor;
      blk[j][1] += m;
      blk[j][2] -= up * K[j] * factor;
      blk[j][3] += um * K[j] * factor;
      blk[j][4] += phi[j] * dPI * factor;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Boundary term of one face for the three local vertices (alpha_boundary; pnp_operator.hh:247-314,
// pb_operator.hh:132-190).  f = DUNE face index of the element, (ax,ay)->(bx,by) the face's
// vertices in element order, j = prescribed flux.  out[i] += j*phi_i*factor for local i = 0..2.
// ---------------------------------------------------------------------------------------------
PNP_HD void boundary_face(int f, double ax, double ay, double bx, double by, double j, const PhysParams& P,
                          double* out) {
  const double len = sqrt((bx - ax) * (bx - ax) + (by - ay) * (by - ay));
  const double tq[2] = {0.21132486540518711775, 0.78867513459481288225};
  for (int q = 0; q < 2; q++) {
    const double t = tq[q];
    double l0, l1;
    if (f == 0) { l0 = t; l1 = 0.0; } else if (f == 1) { l0 = 0.0; l1 = t; } else { l0 = 1.0 - t; l1 = t; }
    const double phi[3] = {1.0 - l0 - l1, l0, l1};
    const double gy = ay + t * (by - ay);
    double factor = 0.5 * len;
    if (P.cylindrical) factor *= gy * 2 * P.PI;
    for (int i = 0; i < 3; i++) out[i] += j * phi[i] * factor;
  }
}

} // namespace pnp
