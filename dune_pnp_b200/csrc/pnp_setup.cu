// pnp_setup.cu -- device-side mesh pipeline: upload, uniform red refinement, locality renumbering,
// vertex-star construction, boundary faces, Dirichlet masks, and the (host-side, test-sized)
// export of the PDELab-shaped CSR pattern/values.
//
// Stands in for GmshReader/GridFactory/UGGrid (pnp_solver_main.cc:82-114), GridFunctionSpace dof
// numbering, constraints() (stationary_pnp.hh:155) and the MatrixContainer pattern
// (stationary_pnp.hh:243-245); semantics per SURVEY.md App. A.4, A.5, A.10.
#include <algorithm>
#include <cub/cub.cuh>
#include <map>

#include "pnp_common.cuh"
#include "pnp_setup_algos.cuh"

namespace pnp {

namespace {

__global__ void k_edge_keys(const int* __restrict__ tri, long nT, uint64_t* __restrict__ keys) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < 3 * nT; i += (long)gridDim.x * blockDim.x)
    keys[i] = tri_edge_key(tri, i);
}
__global__ void k_midpoints(const uint64_t* __restrict__ ukeys, long nE, long nv, double* __restrict__ x,
                            double* __restrict__ y) {
  for (long k = blockIdx.x * (long)blockDim.x + threadIdx.x; k < nE; k += (long)gridDim.x * blockDim.x) {
    int a = (int)(ukeys[k] >> 32), b = (int)(ukeys[k] & 0xffffffffu);
    x[nv + k] = 0.5 * (x[a] + x[b]);
    y[nv + k] = 0.5 * (y[a] + y[b]);
  }
}
__global__ void k_mid_field(const uint64_t* __restrict__ ukeys, long nE, long nv, double* __restrict__ u) {
  for (long k = blockIdx.x * (long)blockDim.x + threadIdx.x; k < nE; k += (long)gridDim.x * blockDim.x) {
    int a = (int)(ukeys[k] >> 32), b = (int)(ukeys[k] & 0xffffffffu);
    u[nv + k] = 0.5 * (u[a] + u[b]);
  }
}
__global__ void k_children(const int* __restrict__ tri, long nT, const uint64_t* __restrict__ ukeys, long nE, long nv,
                           int* __restrict__ out) {
  for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < nT; t += (long)gridDim.x * blockDim.x)
    refine_children(tri, t, ukeys, nE, nv, out + 12 * t);
}
__global__ void k_refine_bnd(const int* __restrict__ ba, const int* __restrict__ bb, const int* __restrict__ ph, long nB,
                             const uint64_t* __restrict__ ukeys, long nE, long nv, int* __restrict__ oa,
                             int* __restrict__ ob, int* __restrict__ op) {
  for (long s = blockIdx.x * (long)blockDim.x + threadIdx.x; s < nB; s += (long)gridDim.x * blockDim.x) {
    int m = (int)(nv + lower_bound_u64(ukeys, nE, edge_key(ba[s], bb[s])));
    oa[2 * s] = ba[s]; ob[2 * s] = m; op[2 * s] = ph[s];
    oa[2 * s + 1] = m; ob[2 * s + 1] = bb[s]; op[2 * s + 1] = ph[s];
  }
}

// ---- renumbering: a vertex's key is the first triangle corner that touches it ----
__global__ void k_first_touch(const int* __restrict__ tri, long nT, int* __restrict__ first) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < 3 * nT; i += (long)gridDim.x * blockDim.x)
    atomicMin(&first[tri[i]], (int)i);
}
__global__ void k_fill_int(int* a, long n, int v) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) a[i] = v;
}
__global__ void k_iota(int* a, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) a[i] = (int)i;
}
__global__ void k_invert_perm(const int* __restrict__ int2ext, long n, int* __restrict__ ext2int) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    ext2int[int2ext[i]] = (int)i;
}
__global__ void k_gather_xy(const int* __restrict__ int2ext, const double* __restrict__ x, const double* __restrict__ y,
                            long n, XY* __restrict__ xy) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int e = int2ext[i];
    xy[i] = XY{x[e], y[e]};
  }
}

// ---- vertex stars from sorted corner records (per-item logic in pnp_setup_algos.cuh) ----
__global__ void k_corner_records(const int* __restrict__ tri, long nT, const int* __restrict__ ext2int,
                                 const double* __restrict__ x, const double* __restrict__ y, uint64_t* __restrict__ keys,
                                 unsigned* __restrict__ pay, int* __restrict__ err) {
  for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < nT; t += (long)gridDim.x * blockDim.x)
    if (!corner_records(tri, t, ext2int, x, y, keys + 3 * t, pay + 3 * t)) atomicExch(err, 1);
}
__global__ void k_rec_start(const uint64_t* __restrict__ keys, long nrec, long nv, int* __restrict__ start) {
  for (long v = blockIdx.x * (long)blockDim.x + threadIdx.x; v <= nv; v += (long)gridDim.x * blockDim.x)
    start[v] = (int)lower_bound_u64(keys, nrec, (uint64_t)v << 32);
}
__global__ void k_ring_count(const uint64_t* __restrict__ keys, const unsigned* __restrict__ pay,
                             const int* __restrict__ start, long nv, int* __restrict__ rowlen, int* __restrict__ err) {
  for (long v = blockIdx.x * (long)blockDim.x + threadIdx.x; v < nv; v += (long)gridDim.x * blockDim.x) {
    int b = start[v], e = start[v + 1], open, bad;
    fan_start(keys, pay, b, e, &open, &bad);
    if (bad) atomicExch(err, 2);
    rowlen[v] = 1 + (e - b) + open;
  }
}
__global__ void k_ring_fill(const uint64_t* __restrict__ keys, const unsigned* __restrict__ pay,
                            const int* __restrict__ start, long nv, const int* __restrict__ rp, unsigned* __restrict__ adj,
                            int* __restrict__ err) {
  for (long v = blockIdx.x * (long)blockDim.x + threadIdx.x; v < nv; v += (long)gridDim.x * blockDim.x)
    if (!ring_fill(keys, pay, start[v], start[v + 1], (int)v, adj + rp[v])) atomicExch(err, 2);
}
// one BFace per boundary segment
__global__ void k_bfaces(const int* __restrict__ ba, const int* __restrict__ bb, const int* __restrict__ ph, long nB,
                         const int* __restrict__ ext2int, const int* __restrict__ rp, const unsigned* __restrict__ adj,
                         int n_own, bool partitioned, BFace* __restrict__ out, int* __restrict__ err) {
  for (long s = blockIdx.x * (long)blockDim.x + threadIdx.x; s < nB; s += (long)gridDim.x * blockDim.x) {
    BFace bf;
    const int a = ext2int[ba[s]], b = ext2int[bb[s]];
    bool ok;
    // the face is reconstructed from the fan of an OWNED end vertex; a face between two ghosts only
    // contributes its Dirichlet flags (v[] stays -1)
    if (a < n_own) ok = boundary_face_of(rp, adj, a, b, &bf);
    else if (b < n_own) ok = boundary_face_of(rp, adj, b, a, &bf);
    else { bf.v[0] = bf.v[1] = bf.v[2] = -1; bf.f = 0; ok = partitioned; }
    if (!ok) atomicExch(err, 3);
    bf.a = a; bf.b = b; bf.phys = ph[s]; bf.seg = (int)s;
    out[s] = bf;
  }
}
__global__ void k_count_open(const int* __restrict__ rp, const unsigned* __restrict__ adj, long nv, int* __restrict__ cnt) {
  int local = 0;
  for (long v = blockIdx.x * (long)blockDim.x + threadIdx.x; v < nv; v += (long)gridDim.x * blockDim.x)
    if (!(adj[rp[v + 1] - 1] & STAR_HAS_TRI)) local++;
  if (local) atomicAdd(cnt, local);
}
__global__ void k_scatter_dmask(const int* __restrict__ vtx, const unsigned char* __restrict__ bits, int n,
                                unsigned char* __restrict__ dmask) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dmask[vtx[i]] = bits[i];
}

// vectors: reference numbering (lexicographic, external vertex ids) <-> internal (vertex-blocked)
__global__ void k_vec_to_internal(const double* __restrict__ lex, const int* __restrict__ int2ext, long nv, int F,
                                  double* __restrict__ blk) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < nv * F; i += (long)gridDim.x * blockDim.x) {
    long v = i / F; int k = (int)(i % F);
    blk[i] = lex[(long)k * nv + int2ext[v]];
  }
}
__global__ void k_vec_to_external(const double* __restrict__ blk, const int* __restrict__ int2ext, long nv, int F,
                                  double* __restrict__ lex) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < nv * F; i += (long)gridDim.x * blockDim.x) {
    long v = i / F; int k = (int)(i % F);
    lex[(long)k * nv + int2ext[v]] = blk[i];
  }
}

struct CubTemp {
  DBuf<unsigned char> buf;
  void* get(size_t bytes) { if (bytes > buf.n) buf.alloc(bytes); return buf.p; }
};

} // namespace

#define LAUNCH(ctx, kern, n, ...)                                                       \
  do { kern<<<grid_for((n), 256), 256, 0, (ctx).stream>>>(__VA_ARGS__); PNP_CHECK_LAUNCH(); (ctx).launches++; } while (0)

void mesh_set(Ctx& c, long nv, const double* x, const double* y, long nT, const int* tri, long nB, const int* ba,
              const int* bb, const int* bphys, long n_own) {
  PNP_REQUIRE(nv > 0 && nT > 0, PNP_E_ARG, "empty mesh");
  for (long i = 0; i < 3 * nT; i++) PNP_REQUIRE(tri[i] >= 0 && tri[i] < nv, PNP_E_MESH, "triangle vertex out of range");
  for (long i = 0; i < nB; i++)
    PNP_REQUIRE(ba[i] >= 0 && ba[i] < nv && bb[i] >= 0 && bb[i] < nv, PNP_E_MESH, "boundary vertex out of range");
  PNP_REQUIRE(n_own > 0 && n_own <= nv, PNP_E_ARG, "owned vertex count out of range");
  c.nv = nv; c.nT = nT; c.nB = nB; c.n_own = n_own;
  c.hier.clear();
  c.halo_nbr.clear(); c.halo_send_ptr.clear(); c.halo_recv_ptr.clear(); c.halo_send_ext.clear();
  // a new mesh drops the registered multigrid levels too (they describe the old one)
  c.mg.clear(); c.mg_gid.release(); c.mg_nglobal = 0; c.mg_aggregated = false; c.mg_replica = nullptr;
  c.invalidate_mesh_objects();
  c.carry.clear();
  c.cx.alloc(nv); c.cy.alloc(nv); c.ctri.alloc(3 * nT); c.cba.alloc(nB); c.cbb.alloc(nB); c.cbphys.alloc(nB);
  c.cx.upload(x, nv, c.stream); c.cy.upload(y, nv, c.stream); c.ctri.upload(tri, 3 * nT, c.stream);
  c.cba.upload(ba, nB, c.stream); c.cbb.upload(bb, nB, c.stream); c.cbphys.upload(bphys, nB, c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
}

static void star_build(Ctx& c, bool renumber);

void mesh_refine(Ctx& c, int levels) {
  PNP_REQUIRE(c.nv > 0, PNP_E_ARG, "no mesh set");
  PNP_REQUIRE(c.n_own == c.nv, PNP_E_ARG, "device refinement works on an unpartitioned mesh (refine before partitioning)");
  CubTemp tmp;
  for (int l = 0; l < levels; l++) {
    const long nT = c.nT, nv = c.nv, nB = c.nB, nk = 3 * nT;
    PNP_REQUIRE(nk < (1l << 31), PNP_E_MESH, "mesh too large to refine");
    // keep this level for the geometric multigrid hierarchy: its star moves out of the context
    if (!c.finalized) star_build(c, true);
    HierLevel hl;
    hl.nv = nv; hl.nslots = c.nslots;
    hl.rp = std::move(c.rp); hl.adj = std::move(c.adj); hl.int2ext = std::move(c.int2ext); hl.ext2int = std::move(c.ext2int);
    c.finalized = false;
    DBuf<uint64_t> keys(nk), sorted(nk), ukeys(nk);
    DBuf<long> d_nE(1);
    LAUNCH(c, k_edge_keys, nk, c.ctri.p, nT, keys.p);
    size_t bytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, bytes, keys.p, sorted.p, (int)nk, 0, 64, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortKeys(tmp.get(bytes), bytes, keys.p, sorted.p, (int)nk, 0, 64, c.stream));
    cub::DeviceSelect::Unique(nullptr, bytes, sorted.p, ukeys.p, d_nE.p, (int)nk, c.stream);
    PNP_CUDA(cub::DeviceSelect::Unique(tmp.get(bytes), bytes, sorted.p, ukeys.p, d_nE.p, (int)nk, c.stream));
    c.launches += 4;
    long nE = 0;
    d_nE.download(&nE, 1, c.stream);
    keys.release(); sorted.release();
    PNP_REQUIRE(nv + nE < (1l << 31), PNP_E_MESH, "mesh too large to refine");
    DBuf<double> nx(nv + nE), ny(nv + nE);
    PNP_CUDA(cudaMemcpyAsync(nx.p, c.cx.p, nv * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
    PNP_CUDA(cudaMemcpyAsync(ny.p, c.cy.p, nv * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
    LAUNCH(c, k_midpoints, nE, ukeys.p, nE, nv, nx.p, ny.p);
    // carried nodal fields (nested iteration): P1 interpolation = the same midpoint rule, field by field
    for (auto& cf : c.carry) {
      const int F = cf.fields;
      DBuf<double> nf((size_t)F * (nv + nE));
      for (int k = 0; k < F; k++) {
        PNP_CUDA(cudaMemcpyAsync(nf.p + (size_t)k * (nv + nE), cf.d.p + (size_t)k * nv, nv * sizeof(double),
                                 cudaMemcpyDeviceToDevice, c.stream));
        LAUNCH(c, k_mid_field, nE, ukeys.p, nE, nv, nf.p + (size_t)k * (nv + nE));
      }
      PNP_CUDA(cudaStreamSynchronize(c.stream));
      cf.d = std::move(nf);
    }
    DBuf<int> ntri(12 * nT), na(2 * nB), nb(2 * nB), np(2 * nB);
    LAUNCH(c, k_children, nT, c.ctri.p, nT, ukeys.p, nE, nv, ntri.p);
    if (nB) LAUNCH(c, k_refine_bnd, nB, c.cba.p, c.cbb.p, c.cbphys.p, nB, ukeys.p, nE, nv, na.p, nb.p, np.p);
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    c.cx = std::move(nx); c.cy = std::move(ny); c.ctri = std::move(ntri);
    c.cba = std::move(na); c.cbb = std::move(nb); c.cbphys = std::move(np);
    c.nv = nv + nE; c.nT = 4 * nT; c.nB = 2 * nB; c.n_own = c.nv;
    hl.nE = nE; hl.edges = std::move(ukeys);
    c.hier.push_back(std::move(hl));
  }
  c.invalidate_mesh_objects();
}

// Stores vectors in reference numbering so that the next mesh_refine() interpolates them to the finer mesh.
void carry_set(Ctx& c, const int* handles, int n) {
  PNP_REQUIRE(c.finalized, PNP_E_ARG, "mesh not finalized");
  c.carry.clear();
  for (int i = 0; i < n; i++) {
    const Vec& v = c.vec(handles[i]);
    Vec cf; cf.fields = v.fields; cf.d.alloc((size_t)v.fields * c.nv);
    LAUNCH(c, k_vec_to_external, c.nv * v.fields, v.d.p, c.int2ext.p, c.nv, v.fields, cf.d.p);
    c.carry.push_back(std::move(cf));
  }
  PNP_CUDA(cudaStreamSynchronize(c.stream));
}
void carry_get(Ctx& c, int i, Vec& out) {
  PNP_REQUIRE(c.finalized, PNP_E_ARG, "mesh not finalized");
  PNP_REQUIRE(i >= 0 && i < (int)c.carry.size(), PNP_E_ARG, "no such carried field");
  PNP_REQUIRE(out.fields == c.carry[i].fields && c.carry[i].d.n == (size_t)out.fields * c.nv, PNP_E_ARG,
              "carried field does not match the vector / current mesh");
  LAUNCH(c, k_vec_to_internal, c.nv * out.fields, c.carry[i].d.p, c.int2ext.p, c.nv, out.fields, out.d.p);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
}

// vertex star of the current mesh: fills c.int2ext/ext2int/xy/rp/adj/nslots
static void star_build(Ctx& c, bool renumber) {
  PNP_REQUIRE(c.nv > 0, PNP_E_ARG, "no mesh set");
  PNP_REQUIRE(c.nv < STAR_MAX_VERTICES, PNP_E_MESH, "more than 2^27 vertices on one GPU");
  const long nv = c.nv, nT = c.nT, nB = c.nB, nrec = 3 * nT, no = c.n_own;
  PNP_REQUIRE(nrec < (1l << 31), PNP_E_MESH, "more than 2^31 triangle corners on one GPU");
  CubTemp tmp;
  size_t bytes = 0;
  c.int2ext.alloc(nv); c.ext2int.alloc(nv);
  if (renumber) {
    // owned vertices are reordered by first touch; ghosts keep their place (grouped by owner rank by the caller)
    DBuf<int> first(nv), first_sorted(nv), ids(nv);
    LAUNCH(c, k_fill_int, nv, first.p, nv, 0x7fffffff);
    LAUNCH(c, k_first_touch, nrec, c.ctri.p, nT, first.p);
    LAUNCH(c, k_iota, nv, ids.p, nv);
    LAUNCH(c, k_iota, nv, c.int2ext.p, nv);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, first.p, first_sorted.p, ids.p, c.int2ext.p, (int)no, 0, 32, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortPairs(tmp.get(bytes), bytes, first.p, first_sorted.p, ids.p, c.int2ext.p, (int)no,
                                            0, 32, c.stream));
    c.launches += 2;
  } else {
    LAUNCH(c, k_iota, nv, c.int2ext.p, nv);
  }
  LAUNCH(c, k_invert_perm, nv, c.int2ext.p, nv, c.ext2int.p);
  c.xy.alloc(nv);
  LAUNCH(c, k_gather_xy, nv, c.int2ext.p, c.cx.p, c.cy.p, nv, c.xy.p);

  DBuf<int> err(1); err.zero(c.stream);
  DBuf<int> start(no + 1), rowlen(no + 1);
  {
    DBuf<uint64_t> keys(nrec), skeys(nrec);
    DBuf<unsigned> pay(nrec), spay(nrec);
    LAUNCH(c, k_corner_records, nT, c.ctri.p, nT, c.ext2int.p, c.cx.p, c.cy.p, keys.p, pay.p, err.p);
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys.p, skeys.p, pay.p, spay.p, (int)nrec, 0, 60, c.stream);
    PNP_CUDA(cub::DeviceRadixSort::SortPairs(tmp.get(bytes), bytes, keys.p, skeys.p, pay.p, spay.p, (int)nrec, 0, 60,
                                            c.stream));
    c.launches += 2;
    keys.release(); pay.release();
    LAUNCH(c, k_rec_start, no + 1, skeys.p, nrec, no, start.p);
    rowlen.zero(c.stream);
    LAUNCH(c, k_ring_count, no, skeys.p, spay.p, start.p, no, rowlen.p, err.p);
    c.rp.alloc(no + 1);
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, rowlen.p, c.rp.p, (int)(no + 1), c.stream);
    PNP_CUDA(cub::DeviceScan::ExclusiveSum(tmp.get(bytes), bytes, rowlen.p, c.rp.p, (int)(no + 1), c.stream));
    c.launches += 1;
    int ns = 0;
    PNP_CUDA(cudaMemcpyAsync(&ns, c.rp.p + no, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PNP_CUDA(cudaStreamSynchronize(c.stream));
    c.nslots = ns;
    c.adj.alloc(c.nslots);
    LAUNCH(c, k_ring_fill, no, skeys.p, spay.p, start.p, no, c.rp.p, c.adj.p, err.p);
  }
  int herr = 0;
  err.download(&herr, 1, c.stream);
  PNP_REQUIRE(herr != 1, PNP_E_MESH, "degenerate triangle (zero area or repeated vertex)");
  PNP_REQUIRE(herr == 0, PNP_E_MESH, "vertex star is not a single fan (non-manifold mesh)");
}

void mesh_finalize(Ctx& c, bool renumber) {
  star_build(c, renumber);
  const long nv = c.nv, nB = c.nB, no = c.n_own;
  DBuf<int> err(1); err.zero(c.stream);
  int herr = 0;

  // boundary faces
  c.d_bfaces.alloc(nB);
  DBuf<int> nopen(1); nopen.zero(c.stream);
  LAUNCH(c, k_count_open, no, c.rp.p, c.adj.p, no, nopen.p);
  if (nB) LAUNCH(c, k_bfaces, nB, c.cba.p, c.cbb.p, c.cbphys.p, nB, c.ext2int.p, c.rp.p, c.adj.p, (int)no, no < nv, c.d_bfaces.p, err.p);
  err.download(&herr, 1, c.stream);
  PNP_REQUIRE(herr == 0, PNP_E_MESH, "a boundary segment (Gmsh line element) is not a boundary edge of the mesh");
  int hopen = 0;
  nopen.download(&hopen, 1, c.stream);
  PNP_REQUIRE(no < nv || hopen == nB, PNP_E_MESH, "boundary face without boundary segment (or duplicate segment)");
  c.bfaces = c.d_bfaces.to_host(c.stream);
  c.dmask.alloc(nv); c.dmask.zero(c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  c.finalized = true; c.constraints_built = false;
  halo_finalize(c);
  if (c.degree >= 2) p2_build(c);
  if (c.params.set) constraints_build(c);
}

// constraints(): face-centre test, both end vertices of a Dirichlet face (SURVEY App. A.5; btype.hh:21-53),
// plus the per-surface flux table (fluxContainer, stationary_pnp.hh:161-186) and the boundary-vertex
// incidence lists the deterministic boundary kernel walks.
void constraints_build(Ctx& c) {
  PNP_REQUIRE(c.finalized, PNP_E_ARG, "mesh not finalized");
  PNP_REQUIRE(c.params.set, PNP_E_ARG, "parameters not set");
  std::map<int, unsigned char> bits;
  std::map<int, std::vector<int>> items;
  for (size_t i = 0; i < c.bfaces.size(); i++) {
    const BFace& b = c.bfaces[i];
    PNP_REQUIRE(b.phys >= 0 && b.phys < c.params.n_surfaces, PNP_E_CONFIG,
                "physical tag of a boundary segment has no [surface_i] section");
    const HostSurface& s = c.params.surfaces[b.phys];
    unsigned char m = 0;
    for (int k = 0; k < 3; k++) if (s.btype[k] == 0) m |= (unsigned char)(1u << k);
    bits[b.a] |= m; bits[b.b] |= m;
    if (b.v[0] < 0) continue; // face between two ghost vertices: flags only
    for (int r = 0; r < 3; r++) if (b.v[r] < c.n_own) items[b.v[r]].push_back((int)i * 4 + r);
  }
  std::vector<int> vtx; std::vector<unsigned char> vb;
  for (auto& kv : bits) { vtx.push_back(kv.first); vb.push_back(kv.second); }
  c.dmask.zero(c.stream);
  if (!vtx.empty()) {
    DBuf<int> dv(vtx.size()); DBuf<unsigned char> db(vb.size());
    dv.upload(vtx.data(), vtx.size(), c.stream); db.upload(vb.data(), vb.size(), c.stream);
    k_scatter_dmask<<<(int)((vtx.size() + 255) / 256), 256, 0, c.stream>>>(dv.p, db.p, (int)vtx.size(), c.dmask.p);
    PNP_CHECK_LAUNCH(); c.launches++;
    PNP_CUDA(cudaStreamSynchronize(c.stream));
  }
  std::vector<int> bv, ptr{0}, it;
  for (auto& kv : items) {
    bv.push_back(kv.first);
    std::vector<int> l = kv.second; std::sort(l.begin(), l.end());
    it.insert(it.end(), l.begin(), l.end());
    ptr.push_back((int)it.size());
  }
  c.n_bv = (int)bv.size();
  c.d_bv.alloc(bv.size()); c.d_bv_ptr.alloc(ptr.size()); c.d_bv_items.alloc(it.size());
  c.d_bv.upload(bv.data(), bv.size(), c.stream); c.d_bv_ptr.upload(ptr.data(), ptr.size(), c.stream);
  c.d_bv_items.upload(it.data(), it.size(), c.stream);
  std::vector<double> surf(3 * (size_t)c.params.n_surfaces);
  for (int i = 0; i < c.params.n_surfaces; i++)
    for (int k = 0; k < 3; k++) surf[3 * i + k] = c.params.surfaces[i].flux[k];
  c.d_surf.alloc(surf.size());
  c.d_surf.upload(surf.data(), surf.size(), c.stream);
  std::vector<unsigned char> sdir(c.params.n_surfaces, 0);
  for (int i = 0; i < c.params.n_surfaces; i++)
    for (int k = 0; k < 3; k++) if (c.params.surfaces[i].btype[k] == 0) sdir[i] |= (unsigned char)(1u << k);
  c.d_surf_dir.alloc(sdir.size());
  c.d_surf_dir.upload(sdir.data(), sdir.size(), c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  if (c.degree >= 2) p2_constraints(c);
  c.constraints_built = true;
}

void vec_upload(Ctx& c, Vec& v, const double* host_lex) {
  PNP_REQUIRE(c.finalized, PNP_E_ARG, "mesh not finalized");
  if (c.degree >= 2) { v.d.upload(host_lex, v.d.n, c.stream); PNP_CUDA(cudaStreamSynchronize(c.stream)); return; } // device layout = the reference's
  const long n = c.nv * v.fields;
  // staging buffer kept between calls: allocating and freeing a vector-sized block per transfer costs more than the copy
  DBuf<double>& tmp = c.io_stage;
  if (tmp.n < (size_t)n) tmp.alloc(n);
  tmp.upload(host_lex, n, c.stream);
  LAUNCH(c, k_vec_to_internal, n, tmp.p, c.int2ext.p, c.nv, v.fields, v.d.p);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
}
// the same conversions between device buffers (linear elements; the p-multigrid of pnp_p2.cu moves vertex values this way)
void vec_from_lex_device(Ctx& c, Vec& v, const double* d_lex) {
  LAUNCH(c, k_vec_to_internal, c.nv * v.fields, d_lex, c.int2ext.p, c.nv, v.fields, v.d.p);
}
void vec_to_lex_device(Ctx& c, const Vec& v, double* d_lex) {
  LAUNCH(c, k_vec_to_external, c.nv * v.fields, v.d.p, c.int2ext.p, c.nv, v.fields, d_lex);
}
void vec_download(Ctx& c, const Vec& v, double* host_lex) {
  if (c.degree >= 2) { v.d.download(host_lex, v.d.n, c.stream); return; }
  const long n = c.nv * v.fields;
  DBuf<double>& tmp = c.io_stage;
  if (tmp.n < (size_t)n) tmp.alloc(n);
  LAUNCH(c, k_vec_to_external, n, v.d.p, c.int2ext.p, c.nv, v.fields, tmp.p);
  tmp.download(host_lex, n, c.stream);
}

// ---- export in the reference's container layout (host side; meant for test-sized meshes) ----
namespace {
struct HostStar {
  std::vector<int> rp, int2ext, ext2int; std::vector<unsigned> adj; std::vector<unsigned char> dmask;
};
HostStar fetch_star(Ctx& c) {
  HostStar h;
  h.rp = c.rp.to_host(c.stream); h.adj = c.adj.to_host(c.stream);
  h.int2ext = c.int2ext.to_host(c.stream); h.ext2int = c.ext2int.to_host(c.stream);
  h.dmask = c.dmask.to_host(c.stream);
  return h;
}
// visits the entries of the PDELab-1.1 pattern in row-major, column-ascending order
template <class Fn> long walk_pattern(Ctx& c, const Operator& op, const HostStar& h, int* rowptr, Fn fn) {
  const int F = op_fields(op.op);
  const long nv = c.nv;
  auto dir = [&](int vint, int k) { return F == 3 ? (h.dmask[vint] >> k) & 1 : (h.dmask[vint] >> op.comp0) & 1; };
  long nnz = 0;
  std::vector<std::pair<int, int>> cols; // (external vertex, slot)
  for (int ki = 0; ki < F; ki++)
    for (long ve = 0; ve < nv; ve++) {
      const int vi = h.ext2int[ve];
      if (rowptr) rowptr[ki * nv + ve] = (int)nnz;
      if (dir(vi, ki)) { fn(nnz, ki, ki, h.rp[vi], true); nnz++; continue; }
      cols.clear();
      for (int s = h.rp[vi]; s < h.rp[vi + 1]; s++) cols.push_back({h.int2ext[h.adj[s] & STAR_VMASK], s});
      std::sort(cols.begin(), cols.end());
      for (int kj = 0; kj < F; kj++)
        for (auto& cs : cols) {
          if (dir(h.ext2int[cs.first], kj)) continue;
          fn(nnz, ki, kj, cs.second, false); nnz++;
        }
    }
  if (rowptr) rowptr[(long)F * nv] = (int)nnz;
  return nnz;
}
} // namespace

long pattern_export(Ctx& c, int op_handle, int* rowptr, int* col) {
  PNP_REQUIRE(c.constraints_built, PNP_E_ARG, "constraints not built");
  PNP_REQUIRE(c.n_own == c.nv, PNP_E_ARG, "pattern export works on an unpartitioned mesh");
  const Operator& op = c.oper(op_handle);
  if (c.degree >= 2) return p2_pattern_export(c, op, rowptr, col);
  HostStar h = fetch_star(c);
  const long nv = c.nv;
  return walk_pattern(c, op, h, rowptr, [&](long k, int ki, int kj, int slot, bool) {
    if (col) col[k] = (int)(kj * nv + h.int2ext[h.adj[slot] & STAR_VMASK]);
    (void)ki;
  });
}

void matrix_export(Ctx& c, int op_handle, const Matrix& A, double* val) {
  PNP_REQUIRE(c.constraints_built, PNP_E_ARG, "constraints not built");
  PNP_REQUIRE(c.n_own == c.nv, PNP_E_ARG, "matrix export works on an unpartitioned mesh");
  const Operator& op = c.oper(op_handle);
  PNP_REQUIRE(A.op == op.op, PNP_E_ARG, "matrix belongs to another operator type");
  if (c.degree >= 2) { PNP_REQUIRE(A.csr_rp, PNP_E_ARG, "matrix not assembled"); A.vals.download(val, A.csr_nnz, c.stream); return; }
  HostStar h = fetch_star(c);
  std::vector<double> v = A.vals.to_host(c.stream);
  const long ns = c.nslots;
  if (A.nplanes == PNP_COMPACT_PLANES) { // expanded as the solver kernels read it: (c+,c+) = L - D, (c-,c-) = L + D, ...
    walk_pattern(c, op, h, nullptr, [&](long k, int ki, int kj, int slot, bool) {
      val[k] = pnp_block_at<PNP_COMPACT_PLANES>(v.data(), ns, slot).at(ki, kj);
    });
    return;
  }
  walk_pattern(c, op, h, nullptr, [&](long k, int ki, int kj, int slot, bool) {
    int pl = op.op == OP_PNP ? pnp_plane(ki, kj) : 0;
    val[k] = pl < 0 ? 0.0 : v[(size_t)pl * ns + slot];
  });
}

// Import of an externally assembled matrix in the container layout of pattern_export() (what `A.base()` of an
// ISTLBCRSMatrixBackend<1,1> matrix holds, stationary_pnp.hh:247): the ISTL-backend-level drop-in --
// ls.apply(A, z, r, red) on a matrix PDELab assembled (instationary_pnp_from_pb_md.hh:188-211).  The pattern must be the
// operator's pattern; entries of the (c+, c-) / (c-, c+) blocks, which the 7-plane layout does not store, must be zero.
void matrix_import(Ctx& c, int op_handle, Matrix& A, const int* rowptr, const int* col, const double* val) {
  PNP_REQUIRE(c.constraints_built, PNP_E_ARG, "constraints not built");
  PNP_REQUIRE(c.n_own == c.nv, PNP_E_ARG, "matrix import works on an unpartitioned mesh");
  PNP_REQUIRE(rowptr && col && val, PNP_E_ARG, "null CSR arrays");
  const Operator& op = c.oper(op_handle);
  PNP_REQUIRE(A.op == op.op, PNP_E_ARG, "matrix belongs to another operator type");
  if (c.degree >= 2) { p2_matrix_import(c, op, A, rowptr, col, val); return; }
  // an arbitrary CSR matrix has no compact form (its diagonal blocks need not share one Laplacian)
  PNP_REQUIRE(A.nplanes == op_planes(op.op), PNP_E_ARG, "matrix import writes the 7-plane PNP layout only");
  HostStar h = fetch_star(c);
  const long ns = c.nslots, nv = c.nv;
  std::vector<double> v((size_t)A.nplanes * ns, 0.0);
  std::vector<int> rp_check((size_t)op_fields(op.op) * nv + 1);
  bool bad_col = false, bad_zero = false;
  const long nnz = walk_pattern(c, op, h, rp_check.data(), [&](long k, int ki, int kj, int slot, bool) {
    if (col[k] != (int)(kj * nv + h.int2ext[h.adj[slot] & STAR_VMASK])) bad_col = true;
    const int pl = op.op == OP_PNP ? pnp_plane(ki, kj) : 0;
    if (pl < 0) { if (val[k] != 0.0) bad_zero = true; }
    else v[(size_t)pl * ns + slot] = val[k];
  });
  for (size_t i = 0; i < rp_check.size(); i++) if (rowptr[i] != rp_check[i]) bad_col = true;
  (void)nnz;
  PNP_REQUIRE(!bad_col, PNP_E_ARG, "CSR pattern differs from the operator's pattern (pnp_pattern_get)");
  PNP_REQUIRE(!bad_zero, PNP_E_ARG, "non-zero entry in a (c+, c-) coupling block: not a PNP Jacobian");
  A.vals.upload(v.data(), v.size(), c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  A.comp0 = op.comp0;
  if (c.last_vals == A.vals.p) c.last_vals = nullptr; // not "the last assembled Jacobian" any more: multigrid uses Galerkin products
}

// dof_perm hook (SURVEY H2): the numbering seen at the boundary is the numbering of the mesh arrays.  A caller whose grid
// numbers vertices differently from the Gmsh file (UGGrid's leaf index after loadBalance(), pnp_solver_main.cc:106-114)
// renumbers the mesh it read with pnp_mesh_read_gmsh: new_index[v] = the caller's index of vertex v.  Element and
// boundary-segment order are kept.
void mesh_renumber(Ctx& c, const int* new_index) {
  PNP_REQUIRE(c.nv > 0 && new_index, PNP_E_ARG, "no mesh set");
  PNP_REQUIRE(c.n_own == c.nv && c.hier.empty() && c.carry.empty(), PNP_E_ARG, "renumber the mesh right after it was set (before refinement / partitioning)");
  const long nv = c.nv;
  std::vector<char> seen((size_t)nv, 0);
  for (long v = 0; v < nv; v++) {
    PNP_REQUIRE(new_index[v] >= 0 && new_index[v] < nv && !seen[new_index[v]], PNP_E_ARG, "vertex permutation is not a bijection");
    seen[new_index[v]] = 1;
  }
  std::vector<double> x = c.cx.to_host(c.stream), y = c.cy.to_host(c.stream), nx((size_t)nv), ny((size_t)nv);
  std::vector<int> tri = c.ctri.to_host(c.stream), ba = c.cba.to_host(c.stream), bb = c.cbb.to_host(c.stream);
  for (long v = 0; v < nv; v++) { nx[new_index[v]] = x[v]; ny[new_index[v]] = y[v]; }
  for (auto& t : tri) t = new_index[t];
  for (auto& t : ba) t = new_index[t];
  for (auto& t : bb) t = new_index[t];
  c.cx.upload(nx.data(), nv, c.stream); c.cy.upload(ny.data(), nv, c.stream); c.ctri.upload(tri.data(), tri.size(), c.stream);
  c.cba.upload(ba.data(), ba.size(), c.stream); c.cbb.upload(bb.data(), bb.size(), c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  c.invalidate_mesh_objects();
}

} // namespace pnp
