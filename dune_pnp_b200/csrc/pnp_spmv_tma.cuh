// pnp_spmv_tma.cuh -- the streaming form of the star SpMV (k_star_op, pnp_spmv.cuh) for levels large enough to fill the
// GPU: one persistent CTA per SM; a producer warp streams the value planes, the column indices, the row pointers and the
// epilogue operands of 128-row tiles into shared memory with 1-D bulk copies (cp.async.bulk, the TMA engine) through a
// ring of mbarrier-guarded stages, while the consumer warps do the products out of shared memory.  The bytes in flight
// no longer sit in registers behind the scoreboard (the plain-load kernel ran at 49 % warps active, 62-64 registers and
// ~14 long-scoreboard stall cycles per issue, profiles/hot_kernels_full_r01d_summary.txt).
//
// Shared memory has no coalescing rule, so a consumer LANE owns a whole ROW (LPR = 1; LPR lanes split a row's slots
// otherwise): no shuffle reduction, no idle lanes on 7-slot rows, one epilogue per row -- the first streaming version
// kept the plain-load kernel's 8-lanes-per-row mapping and was issue-bound at 9 warps per SM (1.83 G warp instructions,
// 30 % issue utilisation, 5.4 ms against the plain-load kernel's 4.0 ms; profiles/spmv_tma_r02_summary.txt).  The x
// gathers of columns inside the window [r0 - 128, r0 + 256) -- 90 % of them with the locality numbering -- are
// shared-memory reads from a staged copy of that part of x; the rest are ordinary loads.
//
// A tile's slots are ONE contiguous range [rp[r0], rp[r0+128]) of every plane, so each plane is one bulk copy; source
// addresses are rounded down and sizes up to the 16-byte granularity bulk copies need (arrays carry 64 bytes of slack,
// DBuf::alloc).  Tiles with more than TMA_CAP slots (average valence > 6.5 over 128 rows: unrefined Gmsh meshes only)
// read their slots with plain loads.
//
// The damped point-block Jacobi epilogue inverts every vertex's 3x3 diagonal block from the diagonal slot that is in
// shared memory anyway, instead of reading a stored inverse (72 B/vertex, 12 % of the smoother's traffic).
#pragma once
#include "pnp_spmv.cuh"

namespace pnp {

constexpr int TMA_TR = 128;                      // rows per tile
constexpr int tma_nw(int lpr) { return TMA_TR * lpr / 32; } // consumer warps for `lpr` lanes per row
// producer warps: one per copy stream of a tile -- NP value planes, column indices, row pointers, x window, and the
// right-hand side / dot operand where the epilogue reads one
constexpr int tma_producers(int np, int epi, int ndot) { return np + 3 + ((epi != EPI_PLAIN || ndot >= 1) ? 1 : 0); }
constexpr int tma_threads(int np, int epi, int ndot, int lpr) { return (tma_nw(lpr) + tma_producers(np, epi, ndot)) * 32; }
constexpr int TMA_CAP = 960;                     // staged slots per tile and plane
constexpr int TMA_MAX_STAGES = 3;
constexpr int TMA_W = 128;                       // rows of x staged on either side of the tile (the gather window)

template <int NP> struct TmaLayout {
  static constexpr int F = NP == 1 ? 1 : 3;
  static constexpr int PLANE = (TMA_CAP + 2) * 8;                    // bytes of one value plane of a stage
  static constexpr int COLS = NP * PLANE;                            // (CAP + 4) column indices
  static constexpr int RP = COLS + (TMA_CAP + 4) * 4;                // (TR + 4) row pointers
  static constexpr int B = RP + (TMA_TR + 4) * 4;                    // F*TR (+2) doubles: right-hand side / dot operand
  // x of the rows [r0 - W, r0 + TR + W): with the locality numbering 90 % of a tile's columns lie in this window
  // (measured on the refined pore mesh), so their gathers are shared-memory reads; the smoother takes the rows' own x
  // from it as well
  static constexpr int XW = B + (F * TMA_TR + 2) * 8;
  static constexpr int STAGE = XW + (F * (TMA_TR + 2 * TMA_W) + 2) * 8;
  static constexpr int YBUF = TMA_TR * F * 8;                        // output staging, per consumer warp a slice
  static constexpr int HEAD = 128;                                   // mbarriers
  static_assert(PLANE % 16 == 0 && COLS % 16 == 0 && RP % 16 == 0 && B % 16 == 0 && XW % 16 == 0 && STAGE % 16 == 0, "bulk copy alignment");
  static constexpr int smem_bytes(int stages) { return HEAD + stages * STAGE + YBUF; }
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  unsigned done;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!done);
}
// global -> shared bulk copy (TMA engine, SASS UBLKCP); completes `bytes` on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// inverse of the diagonal block B = [a b c; d e 0; f 0 g] (pnp_block() of the diagonal slot's NP planes), row `k`; the
// same rule as k_dinv (pnp_amg.cu): a (near-)singular block falls back to the scalar diagonal
template <int NP>
__device__ __forceinline__ void block_inverse_row(const double* dv, int k, double* o) {
  const PnpBlock B = pnp_block<NP>(dv);
  const double a = B.a, b = B.b, c_ = B.c, d = B.d, e = B.e, f = B.f, g = B.g;
  const double det = a * e * g - b * d * g - c_ * e * f;
  const double scale = fabs(a * e * g) + fabs(b * d * g) + fabs(c_ * e * f);
  if (fabs(det) > 1e-12 * scale && scale > 0.0) {
    const double id = 1.0 / det;
    if (k == 0) { o[0] = e * g * id; o[1] = -b * g * id; o[2] = -c_ * e * id; }
    else if (k == 1) { o[0] = -d * g * id; o[1] = (a * g - c_ * f) * id; o[2] = c_ * d * id; }
    else { o[0] = -e * f * id; o[1] = b * f * id; o[2] = (a * e - b * d) * id; }
  } else {
    const double dd = k == 0 ? a : (k == 1 ? e : g);
    const double inv = dd != 0.0 ? 1.0 / dd : 0.0;
    o[0] = k == 0 ? inv : 0.0; o[1] = k == 1 ? inv : 0.0; o[2] = k == 2 ? inv : 0.0;
  }
}

// one slot of a row: y_row += A(row, col) x(col); STAGED: values / column index / x window from the stage
template <int NP, bool STAGED>
__device__ __forceinline__ void slot_product(const StarOpArgs& a, bool ok, int s, const double* sv, const int* vb, const unsigned* sc,
                                             int cbase, const double* sx, int wlo, unsigned wn, double* acc, double* dg) {
  constexpr int F = NP == 1 ? 1 : 3;
  const unsigned c = !ok ? 0u : ((STAGED ? sc[s - cbase] : a.col[s]) & STAR_VMASK);
  const unsigned cw = c - (unsigned)wlo; // (wraps for columns below the window)
  const bool in = cw < wn;
  double x[F], v[NP];
#pragma unroll
  for (int k = 0; k < F; k++) x[k] = !ok ? 0.0 : (in ? sx[F * cw + k] : a.x[(size_t)F * c + k]);
#pragma unroll
  for (int p = 0; p < NP; p++) v[p] = !ok ? 0.0 : (STAGED ? sv[vb[p] + s] : a.vals[(size_t)p * a.stride + s]);
  if (dg) {
#pragma unroll
    for (int p = 0; p < NP; p++) dg[p] = v[p];
  }
  if constexpr (NP == 1) acc[0] += v[0] * x[0];
  else block_mac<NP>(v, x, acc);
}

template <int NP, int EPI, int NDOT, int LPR>
__global__ void __launch_bounds__(tma_threads(NP, EPI, NDOT, LPR), 1) k_star_op_tma(const StarOpArgs a, const int nstages) {
  using L = TmaLayout<NP>;
  constexpr int F = L::F;
  constexpr int TMA_NW = tma_nw(LPR);
  constexpr int RW = 32 / LPR;          // rows per consumer warp and tile
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + TMA_MAX_STAGES;
  unsigned char* stages = smem + L::HEAD;
  double* ybuf = reinterpret_cast<double*>(stages + (size_t)nstages * L::STAGE);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (a.nv + TMA_TR - 1) / TMA_TR;
  const int sp = (int)(a.stride & 1);
  if (threadIdx.x == 0) {
    for (int s = 0; s < nstages; s++) { mbar_init(&full[s], tma_producers(NP, EPI, NDOT)); mbar_init(&empty[s], TMA_NW); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  double dsum[NDOT > 0 ? NDOT : 1];
#pragma unroll
  for (int j = 0; j < (NDOT > 0 ? NDOT : 1); j++) dsum[j] = 0.0;

  if (warp >= TMA_NW) {
    // ---------------- producers: ONE WARP PER COPY STREAM (value plane p, column indices, row pointers, gather window,
    // right-hand side).  Issuing a bulk copy costs a chain of R2UR / ELECT / UBLKCP instructions in a single thread; one
    // thread issuing all eleven copies of a tile needed ~4 300 cycles per tile and paced the whole kernel at 4.1 TB/s
    // whatever the consumers did (profiles/spmv_tma_r02_summary.txt).  Lane 0 of every producer warp issues its copy; the
    // other lanes walk the loop with it (the kernel's closing __syncthreads wants converged warps).
    // The slot range of a tile comes from two row pointers in global memory; a load issued while the bulk copies
    // saturate DRAM takes microseconds, so every lane fetches the boundaries of one of the next 32 tiles, a full batch
    // ahead of their use, and lane 0 picks them up by shuffle.
    const int role = warp - TMA_NW; // 0..NP-1: plane, NP: columns, NP+1: row pointers, NP+2: x window, NP+3: b / w1
    auto load_batch = [&](int batch, int& lo, int& hi) {
      const long tt = blockIdx.x + (long)(batch * 32 + lane) * gridDim.x;
      lo = 0; hi = 0;
      if (tt < ntiles) { lo = a.rp[tt * TMA_TR]; hi = a.rp[min((int)tt * TMA_TR + TMA_TR, a.nv)]; }
    };
    int cur_lo, cur_hi, nxt_lo, nxt_hi;
    load_batch(0, cur_lo, cur_hi);
    load_batch(1, nxt_lo, nxt_hi);
    int t = blockIdx.x;
    for (int it = 0; t < ntiles; t += gridDim.x, it++) {
      if (it > 0 && (it & 31) == 0) { cur_lo = nxt_lo; cur_hi = nxt_hi; load_batch(it / 32 + 1, nxt_lo, nxt_hi); }
      const int lo = __shfl_sync(0xffffffffu, cur_lo, it & 31), hi = __shfl_sync(0xffffffffu, cur_hi, it & 31);
      if (lane == 0) {
        const int stage = it % nstages;
        const unsigned parity = (unsigned)((it / nstages) & 1);
        mbar_wait(&empty[stage], parity ^ 1u);
        unsigned char* st = stages + (size_t)stage * L::STAGE;
        const int r0 = t * TMA_TR, rows = min(TMA_TR, a.nv - r0);
        const bool staged = hi - lo <= TMA_CAP;
        const void* src = nullptr; void* dst = nullptr; unsigned nb = 0;
        if (role < NP) {
          if (staged) {
            const int o = (lo + role * sp) & 1;
            nb = (unsigned)(((hi - lo + o) + 1) & ~1) * 8u;
            src = a.vals + (size_t)role * a.stride + (lo - o); dst = st + role * L::PLANE;
          }
        } else if (role == NP) {
          if (staged) {
            const int lo_c = lo & ~3;
            nb = (unsigned)(((hi - lo_c) + 3) & ~3) * 4u;
            src = a.col + lo_c; dst = st + L::COLS;
          }
        } else if (role == NP + 1) {
          nb = (unsigned)((rows + 1 + 3) & ~3) * 4u;
          src = a.rp + r0; dst = st + L::RP;
        } else if (role == NP + 2) {
          const int wlo = max(r0 - TMA_W, 0), whi = min(r0 + TMA_TR + TMA_W, a.nv);
          nb = (unsigned)((F * (whi - wlo) + 1) & ~1) * 8u;
          src = a.x + (size_t)F * wlo; dst = st + L::XW;
        } else {
          nb = (unsigned)((F * rows + 1) & ~1) * 8u;
          src = (EPI == EPI_PLAIN ? a.w1 : a.b) + (size_t)F * r0; dst = st + L::B;
        }
        if (nb) { mbar_expect_tx(&full[stage], nb); bulk_g2s(dst, src, nb, &full[stage]); }
        else mbar_arrive(&full[stage]);
      }
      __syncwarp();
    }
  } else {
    // ---------------- consumers: lane <-> row (LPR lanes per row) ----------------
    const int sub = lane % LPR;
    double* yw = ybuf + warp * RW * F;
    int t = blockIdx.x;
    for (int it = 0; t < ntiles; t += gridDim.x, it++) {
      const int stage = it % nstages;
      const unsigned parity = (unsigned)((it / nstages) & 1);
      mbar_wait(&full[stage], parity);
      const unsigned char* st = stages + (size_t)stage * L::STAGE;
      const double* sv = reinterpret_cast<const double*>(st);
      const unsigned* sc = reinterpret_cast<const unsigned*>(st + L::COLS);
      const int* srp = reinterpret_cast<const int*>(st + L::RP);
      const double* sb = reinterpret_cast<const double*>(st + L::B);
      const double* sx = reinterpret_cast<const double*>(st + L::XW);
      const int r0 = t * TMA_TR, rows = min(TMA_TR, a.nv - r0);
      const int wlo = max(r0 - TMA_W, 0);
      const unsigned wn = (unsigned)(min(r0 + TMA_TR + TMA_W, a.nv) - wlo); // window rows
      const double* sxo = sx + (size_t)F * (r0 - wlo);                        // the tile's own rows inside the window
      const int lo = srp[0], hi = srp[rows];
      const bool staged = hi - lo <= TMA_CAP; // block-uniform
      const int cbase = lo & ~3;
      int vb[NP]; // plane p, slot s -> sv[vb[p] + s]
#pragma unroll
      for (int p = 0; p < NP; p++) vb[p] = p * (TMA_CAP + 2) - lo + ((lo + p * sp) & 1);
      const int rl = RW * warp + lane / LPR; // row of this lane inside the tile
      const bool valid = rl < rows;
      const int b0 = valid ? srp[rl] : hi, e0 = valid ? srp[rl + 1] : hi;
      double acc[F], dg[NP];
#pragma unroll
      for (int k = 0; k < F; k++) acc[k] = 0.0;
#pragma unroll
      for (int p = 0; p < NP; p++) dg[p] = 0.0;
      const int len = e0 - b0;
      const int maxlen = __reduce_max_sync(0xffffffffu, len);
      if (staged) {
        // The first MAXS slots of the lane in three unrolled phases -- column indices, then ALL x gathers, then the
        // products -- so that the gathers of columns outside the staged window (10 % of the slots, ordinary loads that
        // go to L2 or DRAM while the bulk copies saturate it) are in flight together: taken slot by slot, each of them
        // stalled the warp for a full memory round trip and the consumers, not the feed, paced the kernel
        // (profiles/spmv_tma_r02_summary.txt).  Slot `sub` comes first: for sub == 0 it is the diagonal, whose values
        // the smoother epilogue inverts.
        constexpr int MAXS = (8 + LPR - 1) / LPR;
        unsigned cj[MAXS];
        bool okj[MAXS];
        double xj[MAXS][F];
#pragma unroll
        for (int u = 0; u < MAXS; u++) {
          const int j = sub + u * LPR;
          okj[u] = j < len;
          cj[u] = okj[u] ? (sc[b0 + j - cbase] & STAR_VMASK) : 0u;
        }
#pragma unroll
        for (int u = 0; u < MAXS; u++) {
          const unsigned cw = cj[u] - (unsigned)wlo; // (wraps for columns below the window)
          const bool in = cw < wn;
          const bool ldg = okj[u] && !in, lds = okj[u] && in;
#pragma unroll
          for (int k = 0; k < F; k++) {
            double xg = 0.0, xs = 0.0;
            if (ldg) xg = a.x[(size_t)F * cj[u] + k];
            if (lds) xs = sx[F * cw + k];
            xj[u][k] = in ? xs : xg;
          }
        }
#pragma unroll
        for (int u = 0; u < MAXS; u++) {
          const int s = b0 + sub + u * LPR;
          double v[NP];
#pragma unroll
          for (int p = 0; p < NP; p++) v[p] = okj[u] ? sv[vb[p] + s] : 0.0;
          if (EPI == EPI_JACOBI && u == 0) {
#pragma unroll
            for (int p = 0; p < NP; p++) dg[p] = v[p];
          }
          if constexpr (NP == 1) acc[0] += v[0] * xj[u][0];
          else block_mac<NP>(v, xj[u], acc);
        }
        for (int j = sub + MAXS * LPR; j < maxlen; j += LPR) // rows with more slots (valence > 7)
          slot_product<NP, true>(a, j < len, b0 + j, sv, vb, sc, cbase, sx, wlo, wn, acc, nullptr);
      } else { // over-full tile: slots straight from global memory
        slot_product<NP, false>(a, sub < len, b0 + sub, sv, vb, sc, cbase, sx, wlo, wn, acc, EPI == EPI_JACOBI ? dg : nullptr);
        for (int j = sub + LPR; j < maxlen; j += LPR)
          slot_product<NP, false>(a, j < len, b0 + j, sv, vb, sc, cbase, sx, wlo, wn, acc, nullptr);
      }
      if (LPR > 1) {
#pragma unroll
        for (int k = 0; k < F; k++)
#pragma unroll
          for (int o = LPR / 2; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
      }
      const bool mine = valid && sub == 0;
      double yv[F];
#pragma unroll
      for (int k = 0; k < F; k++) yv[k] = 0.0;
      if (mine) {
        if (EPI == EPI_PLAIN) {
#pragma unroll
          for (int k = 0; k < F; k++) {
            yv[k] = acc[k];
            if (NDOT >= 1) dsum[0] += acc[k] * sb[F * rl + k];
            if (NDOT >= 2) dsum[NDOT >= 2 ? 1 : 0] += acc[k] * acc[k];
          }
        } else if (EPI == EPI_RESIDUAL) {
#pragma unroll
          for (int k = 0; k < F; k++) yv[k] = sb[F * rl + k] - acc[k];
        } else { // damped (point-block) Jacobi step: y = x + omega * D^-1 (b - A x)
          double r[F], z[F];
#pragma unroll
          for (int k = 0; k < F; k++) r[k] = sb[F * rl + k] - acc[k];
          if constexpr (F == 3) {
#pragma unroll
            for (int k = 0; k < F; k++) {
              double o[3];
              block_inverse_row<NP>(dg, k, o);
              z[k] = o[0] * r[0] + o[1] * r[1] + o[2] * r[2];
            }
          } else z[0] = (dg[0] != 0.0 ? 1.0 / dg[0] : 0.0) * r[0];
#pragma unroll
          for (int k = 0; k < F; k++) yv[k] = sxo[F * rl + k] + a.omega * z[k];
        }
      }
      if (sub == 0) {
#pragma unroll
        for (int k = 0; k < F; k++) yw[F * (lane / LPR) + k] = yv[k];
      }
      __syncwarp();
      // this warp's RW*F results are contiguous in y
      {
        const size_t g0 = (size_t)F * (r0 + RW * warp);
        const size_t gend = (size_t)F * a.nv;
#pragma unroll
        for (int i = lane; i < RW * F; i += 32)
          if (g0 + i < gend) a.y[g0 + i] = yw[i];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[stage]);
    }
  }
  if (NDOT > 0) {
    __shared__ double sm[NDOT > 0 ? NDOT : 1][TMA_NW];
#pragma unroll
    for (int j = 0; j < (NDOT > 0 ? NDOT : 1); j++) {
      double s = dsum[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0 && warp < TMA_NW) sm[j][warp] = s;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
      for (int j = 0; j < (NDOT > 0 ? NDOT : 1); j++) {
        double s = lane < TMA_NW ? sm[j][lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) a.partial[(long)blockIdx.x * NDOT + j] = s;
      }
    }
  }
}

// The streaming kernel serves levels with at least two tiles per SM whose arrays sit on 16-byte boundaries; everything
// else (small levels, the Chebyshev epilogue) stays with the plain-load kernel.
inline bool star_op_tma_ok(const Ctx& c, const StarOpArgs& a, int epi) {
  const Tune& t = tune();
  if (!t.tma || epi == EPI_CHEBYSHEV) return false;
  if ((long)a.nv < (t.tma_min_rows >= 0 ? t.tma_min_rows : 2l * TMA_TR * c.sm_count)) return false;
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  return al(a.rp) && al(a.col) && al(a.vals) && al(a.x) && (!a.b || al(a.b)) && (!a.w1 || al(a.w1));
}

inline int star_op_tma_stages() {
  const int v = tune().tma_stages;
  return v < 2 ? 2 : (v > TMA_MAX_STAGES ? TMA_MAX_STAGES : v);
}

template <int NP, int EPI, int NDOT, int LPR>
inline int launch_star_op_tma_lpr(Ctx& c, const StarOpArgs& a) {
  using L = TmaLayout<NP>;
  const int nstages = star_op_tma_stages();
  const int smem = L::smem_bytes(nstages);
  static unsigned long long configured = 0; // per device bit: the attribute is per device and function
  if (!(configured >> (c.device & 63) & 1ull)) {
    PNP_CUDA(cudaFuncSetAttribute(k_star_op_tma<NP, EPI, NDOT, LPR>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::smem_bytes(TMA_MAX_STAGES)));
    configured |= 1ull << (c.device & 63);
  }
  const int ntiles = (a.nv + TMA_TR - 1) / TMA_TR;
  const int grid = ntiles < c.sm_count ? ntiles : c.sm_count;
  k_star_op_tma<NP, EPI, NDOT, LPR><<<grid, tma_threads(NP, EPI, NDOT, LPR), smem, c.stream>>>(a, nstages);
  PNP_CHECK_LAUNCH(); c.launches++;
  return grid;
}
template <int NP, int EPI, int NDOT>
inline int launch_star_op_tma_inst(Ctx& c, const StarOpArgs& a) {
  return tune().tma_lpr == 2 ? launch_star_op_tma_lpr<NP, EPI, NDOT, 2>(c, a) : launch_star_op_tma_lpr<NP, EPI, NDOT, 1>(c, a);
}

// launches the streaming or the plain-load kernel; returns the grid size (number of partial-sum blocks)
// compulsory traffic of one star-op launch: NP value planes + column index per slot; row pointer, x read once and y
// written per row; the epilogue's extra vectors (b; the dot operand; the Chebyshev direction read and written)
template <int EPI, int NDOT>
inline double star_op_bytes(int nplanes, const StarOpArgs& a) {
  const double F = nplanes == 1 ? 1 : 3, nv = a.nv, ns = a.rp ? (double)a.stride : 0.0;
  double b = (8.0 * nplanes + 4.0) * ns + (4.0 + 16.0 * F) * nv;
  if (EPI != EPI_PLAIN) b += 8.0 * F * nv;
  if (EPI == EPI_PLAIN && NDOT >= 1) b += 8.0 * F * nv;
  if (EPI == EPI_CHEBYSHEV) b += 16.0 * F * nv;
  return b;
}
template <int EPI, int NDOT>
inline int launch_star_op_auto(Ctx& c, int nplanes, const StarOpArgs& a, bool fine = true) {
  c.acct(fine ? Ctx::ACC_SPMV_FINE : Ctx::ACC_SPMV_COARSE, star_op_bytes<EPI, NDOT>(nplanes, a));
  if (EPI != EPI_CHEBYSHEV && star_op_tma_ok(c, a, EPI)) {
    constexpr int E = EPI == EPI_CHEBYSHEV ? EPI_PLAIN : EPI; // (never instantiated for Chebyshev)
    return nplanes == 1 ? launch_star_op_tma_inst<1, E, NDOT>(c, a)
         : nplanes == PNP_COMPACT_PLANES ? launch_star_op_tma_inst<PNP_COMPACT_PLANES, E, NDOT>(c, a)
                                         : launch_star_op_tma_inst<7, E, NDOT>(c, a);
  }
  return launch_star_op<EPI, NDOT>(c, nplanes, a);
}

} // namespace pnp
