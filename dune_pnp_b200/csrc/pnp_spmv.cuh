// pnp_spmv.cuh -- the one SpMV kernel of the library (Krylov products and every AMG level operation).
//
// y = A x on the star / plane layout (NP = 1, 5 or 7 value planes) with a fused epilogue.  HBM-bound: per launch it streams NP value planes and
// the column index of every slot once ((8*NP+4)*nslots bytes), the row pointers (4*nv) and writes y (8*F*nv); x is
// gathered (8*F*nv if every entry is fetched from DRAM once -- the locality renumbering keeps the gathers in L1/L2).
//
// Mapping: a warp owns 32 consecutive rows per outer step.  Their row pointers are fetched with ONE coalesced load
// and handed out by shuffles, so the slot loads of all eight 4-row groups are independent of any further memory
// round trip; two groups are processed per inner step (2 x (NP+1) independent loads in flight per lane before the
// dependent x gathers).  8 lanes share a row (rows have ~7 slots: diagonal + 6 neighbours); rows longer than 8
// slots take extra passes.  All lanes of a warp run the same trip counts (shuffles are warp-wide).
#pragma once
#include "pnp_common.cuh"

namespace pnp {

enum : int { EPI_PLAIN = 0, EPI_RESIDUAL = 1, EPI_JACOBI = 2, EPI_CHEBYSHEV = 3 };

struct StarOpArgs {
  const int* rp; const unsigned* col; const double* vals; long stride; int nv;
  const double* x; double* y;
  const double* b = nullptr;      // EPI_RESIDUAL/JACOBI/CHEBYSHEV: right-hand side
  const double* dinv = nullptr;   // inverse diagonal: one value per dof, or (block = 1, 3 fields) the 3x3 inverse of
  int block = 0;                  //   every vertex's diagonal block, row-major, 9 values per vertex (point-block Jacobi)
  double omega = 0.0, c1 = 0.0;   // Jacobi damping / Chebyshev coefficients (omega = c2)
  double* dvec = nullptr;         // Chebyshev direction (in/out)
  const double* w1 = nullptr;     // NDOT >= 1: partial sums of y.w1 ; NDOT == 2: also y.y
  double* partial = nullptr;
  // the same matrix in single precision, NP planes stride32 (a multiple of 4) floats apart: when set, the streaming
  // kernel's residual / smoother step reads these planes instead of `vals` (pnp_spmv_tma.cuh)
  const float* vals32 = nullptr; long stride32 = 0;
};

constexpr int SPMV_BLOCK = 256;
constexpr int SPMV_LANES = 8;

template <int NP> struct SlotData { double v[NP]; unsigned c; };

// acc += B x for the 3x3 block of one slot (NP = 5 or 7 value planes, pnp_block())
template <int NP>
__device__ __forceinline__ void block_mac(const double* v, const double* x, double* acc) {
  const PnpBlock B = pnp_block<NP>(v);
  acc[0] += B.a * x[0] + B.b * x[1] + B.c * x[2];
  acc[1] += B.d * x[0] + B.e * x[1];
  acc[2] += B.f * x[0] + B.g * x[2];
}

template <int NP>
__device__ __forceinline__ void load_slot(const StarOpArgs& a, int s, bool ok, SlotData<NP>& d) {
  if (ok) {
    d.c = a.col[s] & STAR_VMASK;
#pragma unroll
    for (int p = 0; p < NP; p++) d.v[p] = a.vals[p * a.stride + s];
  } else {
    d.c = 0;
#pragma unroll
    for (int p = 0; p < NP; p++) d.v[p] = 0.0;
  }
}
template <int NP>
__device__ __forceinline__ void accumulate(const StarOpArgs& a, const SlotData<NP>& d, bool ok, double* acc) {
  if (!ok) return;
  if (NP == 1) acc[0] += d.v[0] * a.x[d.c];
  else {
    const long c = d.c;
    const double x[3] = {a.x[3 * c], a.x[3 * c + 1], a.x[3 * c + 2]};
    block_mac<NP>(d.v, x, acc);
  }
}

template <int NP, int EPI, int NDOT>
__global__ void __launch_bounds__(SPMV_BLOCK, 4) k_star_op(const StarOpArgs a) {
  constexpr int F = NP == 1 ? 1 : 3;
  constexpr int L = SPMV_LANES, RPW = 32 / L; // 4 rows per group step
  const int lane = threadIdx.x & 31, sub = lane & (L - 1), grp = lane / L;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  double dsum[NDOT > 0 ? NDOT : 1];
#pragma unroll
  for (int j = 0; j < (NDOT > 0 ? NDOT : 1); j++) dsum[j] = 0.0;
  for (int r0 = warp * 32; r0 < a.nv; r0 += nwarps * 32) {
    // row pointers of rows r0 .. r0+32 : lane i holds rp[r0+i]; the end of row r0+31 comes from one extra load
    const int rlo = a.rp[min(r0 + lane, a.nv)];
    const int rend = a.rp[min(r0 + 32, a.nv)];
#pragma unroll 1
    for (int g0 = 0; g0 < 32; g0 += 2 * RPW) {
      if (r0 + g0 >= a.nv) break; // warp-uniform
      int row[2], b[2], e[2];
      SlotData<NP> d[2];
      bool ok[2];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int i = g0 + h * RPW + grp; // 0..31
        row[h] = r0 + i;
        b[h] = __shfl_sync(0xffffffffu, rlo, i);
        const int nxt = __shfl_sync(0xffffffffu, rlo, (i + 1) & 31);
        e[h] = i == 31 ? rend : nxt;
        if (row[h] >= a.nv) e[h] = b[h];
        ok[h] = b[h] + sub < e[h];
        load_slot<NP>(a, b[h] + sub, ok[h], d[h]);
      }
      // Epilogue operands are fetched NOW, together with the slot loads, by the lane that will finish component `sub`
      // of the row (lanes 0..F-1 of the 8-lane group): their addresses only depend on the row, and loading them after
      // the reduction would add one more dependent memory round trip to every step of this latency-bound loop.
      double eb[2], ex[2], ew[2], ed[2], eB[2][3];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        eb[h] = ex[h] = ew[h] = ed[h] = 0.0; eB[h][0] = eB[h][1] = eB[h][2] = 0.0;
        if (sub < F && row[h] < a.nv) {
          const long idx = (long)F * row[h] + sub;
          if (EPI != EPI_PLAIN) eb[h] = a.b[idx];
          if (EPI == EPI_PLAIN && NDOT >= 1) ew[h] = a.w1[idx];
          if (EPI == EPI_JACOBI || EPI == EPI_CHEBYSHEV) {
            ex[h] = a.x[idx];
            if (F == 3 && a.block) {
              const double* B = a.dinv + 9l * row[h] + 3 * sub;
              eB[h][0] = B[0]; eB[h][1] = B[1]; eB[h][2] = B[2];
            } else eB[h][0] = a.dinv[idx];
            if (EPI == EPI_CHEBYSHEV && a.c1 != 0.0) ed[h] = a.dvec[idx];
          }
        }
      }
      double acc[2][F];
#pragma unroll
      for (int h = 0; h < 2; h++) {
#pragma unroll
        for (int k = 0; k < F; k++) acc[h][k] = 0.0;
        accumulate<NP>(a, d[h], ok[h], acc[h]);
      }
      // rows with more than 8 slots (valence > 7): extra passes, trip count made warp-uniform
      int more = max(e[0] - b[0], e[1] - b[1]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) more = max(more, __shfl_xor_sync(0xffffffffu, more, o));
      for (int off = L; off < more; off += L) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const bool okx = b[h] + off + sub < e[h];
          SlotData<NP> dx;
          load_slot<NP>(a, b[h] + off + sub, okx, dx);
          accumulate<NP>(a, dx, okx, acc[h]);
        }
      }
#pragma unroll
      for (int h = 0; h < 2; h++) {
#pragma unroll
        for (int k = 0; k < F; k++)
#pragma unroll
          for (int o = L / 2; o > 0; o >>= 1) acc[h][k] += __shfl_xor_sync(0xffffffffu, acc[h][k], o);
        // every lane of the group now holds the row sums; lane `sub` < F finishes component `sub`
        const double ax = F == 1 ? acc[h][0] : (sub == 0 ? acc[h][0] : (sub == 1 ? acc[h][1 % F] : acc[h][2 % F]));
        const bool mine = sub < F && row[h] < a.nv;
        const long idx = (long)F * row[h] + sub;
        if (EPI == EPI_PLAIN) {
          if (mine) {
            a.y[idx] = ax;
            if (NDOT >= 1) dsum[0] += ax * ew[h];
            if (NDOT >= 2) dsum[NDOT >= 2 ? 1 : 0] += ax * ax;
          }
        } else if (EPI == EPI_RESIDUAL) {
          if (mine) a.y[idx] = eb[h] - ax;
        } else {
          const double rr = eb[h] - ax; // component `sub` of b - A x (lanes sub < F)
          double z;
          if (F == 3) {
            const int g8 = lane & ~(L - 1);
            const double r0v = __shfl_sync(0xffffffffu, rr, g8), r1v = __shfl_sync(0xffffffffu, rr, g8 + 1),
                         r2v = __shfl_sync(0xffffffffu, rr, g8 + 2);
            z = a.block ? eB[h][0] * r0v + eB[h][1] * r1v + eB[h][2] * r2v : eB[h][0] * rr;
          } else z = eB[h][0] * rr;
          if (mine) {
            if (EPI == EPI_JACOBI) a.y[idx] = ex[h] + a.omega * z;
            else { // Chebyshev: d = c1*d + c2*M^-1 (b - A x) ; y = x + d
              const double dn = (a.c1 != 0.0 ? a.c1 * ed[h] : 0.0) + a.omega * z;
              a.dvec[idx] = dn; a.y[idx] = ex[h] + dn;
            }
          }
        }
      }
    }
  }
  if (NDOT > 0) {
    // block-wide sums -> partial[blockIdx.x*NDOT + j]
    __shared__ double sm[NDOT > 0 ? NDOT : 1][SPMV_BLOCK / 32];
    const int w = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < (NDOT > 0 ? NDOT : 1); j++) {
      double s = dsum[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) sm[j][w] = s;
    }
    __syncthreads();
    if (w == 0) {
#pragma unroll
      for (int j = 0; j < (NDOT > 0 ? NDOT : 1); j++) {
        double s = lane < SPMV_BLOCK / 32 ? sm[j][lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) a.partial[(long)blockIdx.x * NDOT + j] = s;
      }
    }
  }
}

inline int star_op_grid(const Ctx& c, long nv) {
  const long warps = (nv + 31) / 32;
  long blocks = (warps * 32 + SPMV_BLOCK - 1) / SPMV_BLOCK;
  const long cap = (long)c.sm_count * 8;
  return (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

// launches k_star_op<NP,EPI,NDOT>; returns the grid size (number of partial-sum blocks)
template <int EPI, int NDOT>
inline int launch_star_op(Ctx& c, int nplanes, const StarOpArgs& a) {
  const int grid = star_op_grid(c, a.nv);
  if (nplanes == 1) k_star_op<1, EPI, NDOT><<<grid, SPMV_BLOCK, 0, c.stream>>>(a);
  else if (nplanes == PNP_COMPACT_PLANES) k_star_op<PNP_COMPACT_PLANES, EPI, NDOT><<<grid, SPMV_BLOCK, 0, c.stream>>>(a);
  else k_star_op<7, EPI, NDOT><<<grid, SPMV_BLOCK, 0, c.stream>>>(a);
  PNP_CHECK_LAUNCH(); c.launches++;
  return grid;
}

} // namespace pnp
