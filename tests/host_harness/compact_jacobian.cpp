// compact_jacobian.cpp -- TEST INFRASTRUCTURE: the exact PNP Jacobian rows of one triangle in the 7-plane and in the
// compact 5-plane layout (dune_pnp_b200/csrc/pnp_elem.cuh), and the rule that picks the layout (pnp_star.cuh), for
// tests/test_host_compact_jacobian.py.  Compiled there with g++ -ffp-contract=off; never linked into the product.
#include "../../dune_pnp_b200/csrc/pnp_star.cuh"

using namespace pnp;

namespace {
template <int I>
void rows(const Geo& G, const PhysParams& P, const double (*xl)[3], double* full, double* compact, double* expanded) {
  double b7[3][7] = {}, b5[3][PNP_COMPACT_PLANES] = {}, aux[1][3] = {};
  jac_rows_exact<OP_PNP, I>(G, P, xl, aux, b7);
  jac_rows_exact_compact<I>(G, P, xl, b5);
  for (int j = 0; j < 3; j++) {
    const PnpBlock B = pnp_block<PNP_COMPACT_PLANES>(b5[j]);
    const double e[7] = {B.a, B.b, B.c, B.d, B.e, B.f, B.g};
    for (int p = 0; p < 7; p++) { full[7 * j + p] = b7[j][p]; expanded[7 * j + p] = e[p]; }
    for (int p = 0; p < PNP_COMPACT_PLANES; p++) compact[PNP_COMPACT_PLANES * j + p] = b5[j][p];
  }
}
} // namespace

extern "C" {

// xy[6]: the triangle's vertices in element-local order; xl[9]: field k at local vertex i (xl[3k + i]);
// phys[5] = {PI, l_b, c0, valency, cylindrical}; I: the local test function.  Per column vertex j:
// full[7j + p] = 7-plane row, compact[5j + p] = compact row, expanded[7j + p] = the compact row's block entries a..g
void hc_rows(const double* xy, const double* xl, const double* phys, int I, double* full, double* compact, double* expanded) {
  const Geo G = make_geo(xy[0], xy[1], xy[2], xy[3], xy[4], xy[5]);
  PhysParams P;
  P.PI = phys[0]; P.l_b = phys[1]; P.c0 = phys[2]; P.valency = phys[3]; P.cylindrical = (int)phys[4];
  double x[3][3];
  for (int k = 0; k < 3; k++)
    for (int i = 0; i < 3; i++) x[k][i] = xl[3 * k + i];
  if (I == 0) rows<0>(G, P, x, full, compact, expanded);
  else if (I == 1) rows<1>(G, P, x, full, compact, expanded);
  else rows<2>(G, P, x, full, compact, expanded);
}

int hc_jacobian_planes(int mode, int degree, int solver_ok, const int* btype, int n_surfaces) {
  return pnp_jacobian_planes(mode, degree, solver_ok != 0, btype, n_surfaces);
}

} // extern "C"
