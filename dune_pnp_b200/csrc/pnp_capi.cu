// pnp_capi.cu -- extern "C" entry points declared in include/pnp_b200.h.  No exception leaves this file.
#include <cuda_profiler_api.h>

#include <cstring>

#include "pnp_common.cuh"

namespace pnp {
int newton_apply(Ctx&, const Operator&, Vec&, Solver&, const pnp_newton_opts&, pnp_newton_result&);
int amg_graph_state(const Solver&); // pnp_amg.cu
LinResult slp_apply(Ctx&, const Operator&, Vec&, Solver&, double, int, double);
int onestep_apply(Ctx&, int, const Operator&, const Operator&, Solver&, double, Vec&, Vec&, Vec&, double, int, double, LinResult*);
int pnp_context_planes(const Ctx&, int jac_mode, bool solver_ok); // pnp_newton.cu
namespace {
__global__ void k_fill(double* x, long n, double v) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) x[i] = v;
}
__global__ void k_pack3(const double* a, const double* b, const double* c, long nv, double* out) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < nv; i += (long)gridDim.x * blockDim.x) {
    out[3 * i] = a[i]; out[3 * i + 1] = b[i]; out[3 * i + 2] = c[i];
  }
}
__global__ void k_extract(const double* in, long nv, int field, double* out) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < nv; i += (long)gridDim.x * blockDim.x) out[i] = in[3 * i + field];
}
void to_lin(const LinResult& lr, pnp_lin_result* out) {
  if (!out) return;
  out->converged = lr.converged; out->iterations = lr.iterations; out->reduction = lr.reduction;
  out->conv_rate = lr.conv_rate; out->seconds = lr.seconds; out->status = lr.status;
}
} // namespace
} // namespace pnp

using namespace pnp;


#define API_BEGIN(ctx)                                  \
  if (!(ctx)) return PNP_E_ARG;                         \
  Ctx& c = (ctx)->c;                                    \
  try {                                                 \
    PNP_CUDA(cudaSetDevice(c.device));
#define API_END                                                      \
    return PNP_OK;                                                   \
  } catch (const pnp::Error& e) { c.err = e.what(); return e.code; } \
  catch (const std::exception& e) { c.err = e.what(); return PNP_E_ARG; }

namespace pnp {
Ctx* ctx_make_owned_child(Ctx& p) {
  pnp_ctx* h = new pnp_ctx;
  h->c.device = p.device; h->c.stream = p.stream; h->c.owns_stream = false; h->c.sm_count = p.sm_count;
  h->c.params = p.params;
  h->c.parent = &p; p.children.push_back(&h->c);
  p.owned_children.push_back(h);
  return &h->c;
}
void ctx_destroy_owned_child(Ctx& p, Ctx* child) {
  for (size_t i = 0; i < p.owned_children.size(); i++) {
    pnp_ctx* h = (pnp_ctx*)p.owned_children[i];
    if (&h->c != child) continue;
    p.owned_children.erase(p.owned_children.begin() + i);
    pnp_ctx_destroy(h);
    return;
  }
}
} // namespace pnp

extern "C" {

pnp_status pnp_ctx_create(int device, pnp_ctx** out) {
  if (!out) return PNP_E_ARG;
  *out = nullptr;
  int ndev = 0;
  // no CPU fallback: without a CUDA device there is no context
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return PNP_E_CUDA;
  pnp_ctx* h = new pnp_ctx;
  h->c.device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreate(&h->c.stream) != cudaSuccess) { delete h; return PNP_E_CUDA; }
  cudaDeviceGetAttribute(&h->c.sm_count, cudaDevAttrMultiProcessorCount, device);
  *out = h;
  return PNP_OK;
}
pnp_status pnp_ctx_create_child(pnp_ctx* parent, pnp_ctx** out) {
  if (!parent || !out) return PNP_E_ARG;
  pnp_ctx* h = new pnp_ctx;
  Ctx& p = parent->c;
  h->c.device = p.device; h->c.stream = p.stream; h->c.owns_stream = false; h->c.sm_count = p.sm_count;
  h->c.rank = p.rank; h->c.world = p.world; h->c.nccl = p.nccl;
  h->c.params = p.params;
  h->c.parent = &p; p.children.push_back(&h->c);
  *out = h;
  return PNP_OK;
}
// Lifetime of child contexts: a child may be destroyed before its parent (the parent then forgets every multigrid level
// from that child downwards, and a multigrid built on them is rebuilt at its next use); a parent destroyed first
// orphans its children (they lose the borrowed stream and communicator and must only be destroyed afterwards).
void pnp_ctx_destroy(pnp_ctx* ctx) {
  if (!ctx) return;
  Ctx& c = ctx->c;
  cudaSetDevice(c.device);
  if (c.parent) {
    Ctx& p = *c.parent;
    for (size_t i = 0; i < p.children.size(); i++) if (p.children[i] == &c) { p.children.erase(p.children.begin() + i); break; }
    for (size_t i = 0; i < p.mg.size(); i++) if (p.mg[i].lc == &c) { p.mg.resize(i); p.mg_gid.release(); p.mg_nglobal = 0; p.mg_replica = nullptr; break; }
    if (p.mg_replica == &c) { p.mg_replica = nullptr; p.mg_gid.release(); p.mg_nglobal = 0; }
    p.mg_epoch++;
  }
  if (c.stream) cudaStreamSynchronize(c.stream);
  // CUDA graphs that captured NCCL operations must be gone before their communicator is torn down (the tear-down waits
  // for them otherwise: a finished multi-GPU run never exited): drop every solver -- this context's and its children's,
  // whose multigrid objects may hold such graphs -- first
  c.solvers.clear();
  { // levels pnp_partition_build created belong to this context
    std::vector<void*> owned;
    owned.swap(c.owned_children);
    for (void* h : owned) pnp_ctx_destroy((pnp_ctx*)h);
  }
  for (Ctx* k : c.children) { k->solvers.clear(); k->parent = nullptr; k->stream = nullptr; k->nccl = nullptr; }
  if (c.h_red) cudaFreeHost(c.h_red);
  for (cudaEvent_t e : c.prof_ev) cudaEventDestroy(e);
  if (c.tm0) cudaEventDestroy(c.tm0);
  if (c.tm1) cudaEventDestroy(c.tm1);
  if (c.owns_comm) comm_destroy(c);
  cudaStream_t s = c.owns_stream ? c.stream : nullptr;
  delete ctx;
  if (s) cudaStreamDestroy(s);
}
pnp_status pnp_mg_push_level(pnp_ctx* ctx, pnp_ctx* child, const int* par0, const int* par1) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.degree == 1, PNP_E_ARG, "built for linear elements only");
  PNP_REQUIRE(child && par0 && par1, PNP_E_ARG, "null arguments");
  Ctx& f = c.mg.empty() ? c : *c.mg.back().lc;   // the next finer level
  Ctx& k = child->c;
  PNP_REQUIRE(f.finalized && k.finalized, PNP_E_ARG, "both levels must be finalized");
  std::vector<int> fi2e = f.int2ext.to_host(c.stream), ke2i = k.ext2int.to_host(c.stream);
  std::vector<int> p0(f.nv), p1(f.nv);
  for (long i = 0; i < f.nv; i++) {
    const int e = fi2e[i];
    PNP_REQUIRE(par0[e] < k.nv && par1[e] < k.nv, PNP_E_ARG, "parent index out of range");
    p0[i] = par0[e] >= 0 ? ke2i[par0[e]] : -1;
    p1[i] = par1[e] >= 0 ? ke2i[par1[e]] : -1;
  }
  MgLevelRef r; r.lc = &k;
  r.par0.alloc(f.nv); r.par1.alloc(f.nv);
  r.par0.upload(p0.data(), f.nv, c.stream); r.par1.upload(p1.data(), f.nv, c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  c.mg.push_back(std::move(r));
  c.mg_epoch++;
  API_END
}
pnp_status pnp_mg_set_coarse_aggregates(pnp_ctx* ctx, const int* agg, long n_aggregates) {
  const pnp_status st = pnp_mg_set_coarse_global(ctx, agg, n_aggregates);
  if (st == PNP_OK) ctx->c.mg_aggregated = true;
  return st;
}
pnp_status pnp_mg_set_coarse_global(pnp_ctx* ctx, const int* gid, long n_global) {
  API_BEGIN(ctx)
  c.mg_aggregated = false; c.mg_replica = nullptr;
  PNP_REQUIRE(!c.mg.empty() && gid && n_global > 0, PNP_E_ARG, "no multigrid level pushed");
  Ctx& k = *c.mg.back().lc;
  std::vector<int> i2e = k.int2ext.to_host(c.stream), g(k.nv);
  for (long i = 0; i < k.nv; i++) { g[i] = gid[i2e[i]]; PNP_REQUIRE(g[i] >= 0 && g[i] < n_global, PNP_E_ARG, "global index out of range"); }
  c.mg_gid.alloc(k.nv); c.mg_gid.upload(g.data(), k.nv, c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  c.mg_nglobal = n_global; c.mg_epoch++;
  API_END
}
pnp_status pnp_mg_set_coarse_replica(pnp_ctx* ctx, pnp_ctx* replica, const int* gid, long n_global) {
  API_BEGIN(ctx)
  c.mg_aggregated = false; c.mg_replica = nullptr;
  PNP_REQUIRE(!c.mg.empty() && gid && n_global > 0 && replica, PNP_E_ARG, "no multigrid level pushed / null arguments");
  Ctx& k = *c.mg.back().lc;
  Ctx& r = replica->c;
  PNP_REQUIRE(r.finalized && r.n_own == r.nv && r.nv == n_global, PNP_E_ARG, "the replica must hold the whole coarsest mesh, finalized");
  std::vector<int> i2e = k.int2ext.to_host(c.stream), re2i = r.ext2int.to_host(c.stream), g(k.nv);
  for (long i = 0; i < k.nv; i++) {
    const int gi = gid[i2e[i]];
    PNP_REQUIRE(gi >= 0 && gi < n_global, PNP_E_ARG, "global index out of range");
    g[i] = re2i[gi]; // straight into the replica's internal numbering: gathered vectors are the replica's vectors
  }
  c.mg_gid.alloc(k.nv); c.mg_gid.upload(g.data(), k.nv, c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  c.mg_nglobal = n_global; c.mg_replica = &r; c.mg_epoch++;
  API_END
}
pnp_status pnp_profile_spmv(pnp_ctx* ctx, int enable) {
  API_BEGIN(ctx) c.prof = enable != 0; c.prof_used = 0; API_END
}
pnp_status pnp_profile_spmv_get(pnp_ctx* ctx, long* launches, double* total_ms) {
  API_BEGIN(ctx)
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  for (int k = 0; k < 3; k++) { if (launches) launches[k] = 0; if (total_ms) total_ms[k] = 0; }
  for (size_t i = 0; i + 1 < c.prof_used; i += 2) {
    float t = 0; PNP_CUDA(cudaEventElapsedTime(&t, c.prof_ev[i], c.prof_ev[i + 1]));
    const int k = c.prof_kind[i / 2];
    if (launches) launches[k]++;
    if (total_ms) total_ms[k] += t;
  }
  API_END
}
pnp_status pnp_profile_bytes(pnp_ctx* ctx, int reset, double* out6) {
  API_BEGIN(ctx)
  for (int k = 0; k < Ctx::ACC_N; k++) { if (out6) out6[k] = c.alg_bytes[k]; if (reset) c.alg_bytes[k] = 0; }
  API_END
}
pnp_status pnp_profiler_range(pnp_ctx* ctx, int start) {
  API_BEGIN(ctx)
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  if (start) cudaProfilerStart(); else cudaProfilerStop();
  API_END
}
pnp_status pnp_timer_start(pnp_ctx* ctx) {
  API_BEGIN(ctx)
  if (!c.tm0) { PNP_CUDA(cudaEventCreate(&c.tm0)); PNP_CUDA(cudaEventCreate(&c.tm1)); }
  PNP_CUDA(cudaEventRecord(c.tm0, c.stream));
  API_END
}
pnp_status pnp_timer_stop(pnp_ctx* ctx, double* ms) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.tm0 && ms, PNP_E_ARG, "timer not started");
  PNP_CUDA(cudaEventRecord(c.tm1, c.stream));
  PNP_CUDA(cudaEventSynchronize(c.tm1));
  float t = 0; PNP_CUDA(cudaEventElapsedTime(&t, c.tm0, c.tm1));
  *ms = t;
  API_END
}
pnp_status pnp_tune(const char* name, double value) {
  if (!name) return PNP_E_ARG;
  const std::string n(name);
  Tune& t = tune();
  if (n == "tma") t.tma = value != 0;
  else if (n == "tma_stages") t.tma_stages = (int)value;
  else if (n == "tma_lpr") t.tma_lpr = (int)value;
  else if (n == "graph") t.graph = value != 0;
  else if (n == "fd_warp") t.fd_warp = value != 0;
  else if (n == "jac_compact") t.jac_compact = value != 0;
  else if (n == "matrix_compact") t.matrix_compact = value != 0;
  else if (n == "p2_chunk") t.p2_chunk = (long)value;
  else if (n == "tma_min_rows") t.tma_min_rows = (long)value;
  else if (n == "mg_f32_min_rows") t.mg_f32_min_rows = value > 9e18 ? (long)9e18 : (long)value;
  else return PNP_E_ARG;
  return PNP_OK;
}
const char* pnp_last_error(pnp_ctx* ctx) { return ctx ? ctx->c.err.c_str() : "null context"; }
long pnp_launch_count(pnp_ctx* ctx) { return ctx ? ctx->c.launches : 0; }

pnp_status pnp_mesh_set(pnp_ctx* ctx, long nv, const double* x, const double* y, long nT, const int* tri, long nB,
                        const int* ba, const int* bb, const int* bphys) {
  API_BEGIN(ctx) mesh_set(c, nv, x, y, nT, tri, nB, ba, bb, bphys, nv); API_END
}
pnp_status pnp_mesh_set_local(pnp_ctx* ctx, long nv, long n_own, const double* x, const double* y, long nT, const int* tri,
                              long nB, const int* ba, const int* bb, const int* bphys) {
  API_BEGIN(ctx) mesh_set(c, nv, x, y, nT, tri, nB, ba, bb, bphys, n_own); API_END
}
pnp_status pnp_comm_unique_id(char* out128) {
  try { comm_unique_id(out128); return PNP_OK; } catch (...) { return PNP_E_CUDA; }
}
pnp_status pnp_comm_init(pnp_ctx* ctx, int rank, int world, const char* unique_id128) {
  API_BEGIN(ctx) comm_init(c, rank, world, unique_id128); API_END
}
pnp_status pnp_comm_init_file(pnp_ctx* ctx, int rank, int world, const char* path) {
  API_BEGIN(ctx)
  PNP_REQUIRE(world == 1 || path, PNP_E_ARG, "null rendezvous path");
  comm_bootstrap_file(c, rank, world, path ? path : "");
  API_END
}
pnp_status pnp_comm_allgatherv(pnp_ctx* ctx, const void* send, long nbytes, void* recv, long cap, long* counts) {
  API_BEGIN(ctx)
  PNP_REQUIRE(nbytes >= 0 && counts && (nbytes == 0 || send), PNP_E_ARG, "bad all-gather arguments");
  std::vector<long> cnt;
  std::vector<unsigned char> all = comm_allgatherv(c, send, nbytes, cnt);
  for (int r = 0; r < c.world; r++) counts[r] = cnt[r];
  if (recv) {
    PNP_REQUIRE((long)all.size() <= cap, PNP_E_ARG, "receive buffer too small");
    std::memcpy(recv, all.data(), all.size());
  }
  API_END
}
pnp_status pnp_halo_set(pnp_ctx* ctx, int n_nbr, const int* nbr, const int* send_ptr, const int* send_idx, const int* recv_ptr) {
  API_BEGIN(ctx) halo_set(c, n_nbr, nbr, send_ptr, send_idx, recv_ptr); API_END
}
pnp_status pnp_halo_exchange(pnp_ctx* ctx, int vec_handle) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.degree == 1, PNP_E_ARG, "built for linear elements only");
  halo_exchange(c, c.vec(vec_handle).d.p, c.vec(vec_handle).fields);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}
pnp_status pnp_mesh_read_gmsh(pnp_ctx* ctx, const char* path) {
  API_BEGIN(ctx)
  std::vector<double> x, y; std::vector<int> tri, ba, bb, ph;
  read_gmsh_file(path, x, y, tri, ba, bb, ph);
  mesh_set(c, (long)x.size(), x.data(), y.data(), (long)tri.size() / 3, tri.data(), (long)ba.size(), ba.data(), bb.data(),
           ph.data(), (long)x.size());
  API_END
}
pnp_status pnp_mesh_refine(pnp_ctx* ctx, int levels) { API_BEGIN(ctx) mesh_refine(c, levels); API_END }
pnp_status pnp_carry_set(pnp_ctx* ctx, const int* vec_handles, int n) { API_BEGIN(ctx) PNP_REQUIRE(c.degree == 1, PNP_E_ARG, "built for linear elements only"); carry_set(c, vec_handles, n); API_END }
pnp_status pnp_carry_get(pnp_ctx* ctx, int index, int vec_handle) { API_BEGIN(ctx) PNP_REQUIRE(c.degree == 1, PNP_E_ARG, "built for linear elements only"); carry_get(c, index, c.vec(vec_handle)); API_END }
pnp_status pnp_carry_set_host(pnp_ctx* ctx, int fields, const double* host) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.degree == 1, PNP_E_ARG, "built for linear elements only");
  PNP_REQUIRE(c.nv > 0 && fields >= 1 && host, PNP_E_ARG, "no mesh / bad field count");
  Vec cf; cf.fields = fields; cf.d.alloc((size_t)fields * c.nv);
  cf.d.upload(host, (size_t)fields * c.nv, c.stream);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  c.carry.clear();
  c.carry.push_back(std::move(cf));
  API_END
}
pnp_status pnp_carry_get_host(pnp_ctx* ctx, int index, double* host) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.degree == 1, PNP_E_ARG, "built for linear elements only");
  PNP_REQUIRE(index >= 0 && index < (int)c.carry.size() && host, PNP_E_ARG, "no such carried field");
  c.carry[index].d.download(host, c.carry[index].d.n, c.stream);
  API_END
}
pnp_status pnp_mesh_finalize(pnp_ctx* ctx, int renumber) { API_BEGIN(ctx) mesh_finalize(c, renumber != 0); API_END }
pnp_status pnp_mesh_sizes(pnp_ctx* ctx, long* nv, long* nT, long* nB, long* nslots) {
  API_BEGIN(ctx)
  if (nv) *nv = c.nv;
  if (nT) *nT = c.nT; if (nB) *nB = c.nB; if (nslots) *nslots = c.finalized ? c.nslots : 0;
  API_END
}
pnp_status pnp_mesh_get(pnp_ctx* ctx, double* x, double* y, int* tri, int* ba, int* bb, int* bphys) {
  API_BEGIN(ctx)
  if (x) c.cx.download(x, c.nv, c.stream);
  if (y) c.cy.download(y, c.nv, c.stream);
  if (tri) c.ctri.download(tri, 3 * c.nT, c.stream);
  if (ba) c.cba.download(ba, c.nB, c.stream);
  if (bb) c.cbb.download(bb, c.nB, c.stream);
  if (bphys) c.cbphys.download(bphys, c.nB, c.stream);
  API_END
}

pnp_status pnp_params_set(pnp_ctx* ctx, const double* sys, const double* surf) {
  API_BEGIN(ctx)
  PNP_REQUIRE(sys && (sys[0] == 0 || surf), PNP_E_ARG, "null parameter arrays");
  HostParams p;
  p.n_surfaces = (int)sys[0]; p.cylindrical = sys[1] != 0; p.l_b = sys[2]; p.c0 = sys[3]; p.PI = sys[4];
  p.linearSolverIterations = (int)sys[5]; p.newtonReassembleThreshold = sys[6]; p.newtonReduction = sys[7];
  p.newtonMinLinearReduction = sys[8]; p.newtonMaxIterations = sys[9]; p.newtonLineSearchMaxIteration = sys[10];
  p.tau = sys[11]; p.nSteps = (int)sys[12]; p.outputFreq = (int)sys[13]; p.potentialUpdateFreq = (int)sys[14];
  p.verbosity = (int)sys[15];
  PNP_REQUIRE(p.n_surfaces >= 0, PNP_E_CONFIG, "n_surfaces must be non-negative");
  p.surfaces.assign(p.n_surfaces, HostSurface());
  for (int i = 0; i < p.n_surfaces; i++)
    for (int k = 0; k < 3; k++) {
      p.surfaces[i].btype[k] = (int)surf[9 * i + 3 * k];
      p.surfaces[i].flux[k] = surf[9 * i + 3 * k + 1];
      p.surfaces[i].dval[k] = surf[9 * i + 3 * k + 2];
    }
  p.set = true;
  c.params = p;
  c.constraints_built = false;
  if (c.finalized) constraints_build(c);
  API_END
}
pnp_status pnp_params_read(pnp_ctx* ctx, const char* cfg_path) {
  API_BEGIN(ctx)
  read_config_file(cfg_path, c.params);
  c.constraints_built = false;
  if (c.finalized) constraints_build(c);
  API_END
}
pnp_status pnp_params_get(pnp_ctx* ctx, double* sys, double* surf, char* meshfile, int meshfile_cap) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.params.set, PNP_E_ARG, "parameters not set");
  const HostParams& p = c.params;
  const double v[16] = {(double)p.n_surfaces, (double)p.cylindrical, p.l_b, p.c0, p.PI, (double)p.linearSolverIterations,
                        p.newtonReassembleThreshold, p.newtonReduction, p.newtonMinLinearReduction, p.newtonMaxIterations,
                        p.newtonLineSearchMaxIteration, p.tau, (double)p.nSteps, (double)p.outputFreq,
                        (double)p.potentialUpdateFreq, (double)p.verbosity};
  if (sys) std::memcpy(sys, v, sizeof v);
  if (surf)
    for (int i = 0; i < p.n_surfaces; i++)
      for (int k = 0; k < 3; k++) {
        surf[9 * i + 3 * k] = p.surfaces[i].btype[k];
        surf[9 * i + 3 * k + 1] = p.surfaces[i].flux[k];
        surf[9 * i + 3 * k + 2] = p.surfaces[i].dval[k];
      }
  if (meshfile && meshfile_cap > 0) { std::strncpy(meshfile, p.meshfile.c_str(), meshfile_cap - 1); meshfile[meshfile_cap - 1] = 0; }
  API_END
}
pnp_status pnp_constraints_build(pnp_ctx* ctx) { API_BEGIN(ctx) constraints_build(c); API_END }

pnp_status pnp_operator_create(pnp_ctx* ctx, int op, int comp0, int* handle) {
  API_BEGIN(ctx)
  PNP_REQUIRE(op >= PNP_OP_PB && op <= PNP_OP_PNP && comp0 >= 0 && comp0 < 3 && handle, PNP_E_ARG, "bad operator arguments");
  auto o = std::make_unique<Operator>();
  o->op = op; o->comp0 = comp0;
  c.ops.push_back(std::move(o));
  *handle = (int)c.ops.size() - 1;
  API_END
}
pnp_status pnp_operator_set_coefficient(pnp_ctx* ctx, int h, int which, int vec_handle) {
  API_BEGIN(ctx)
  PNP_REQUIRE(which == 0 || which == 1, PNP_E_ARG, "coefficient index must be 0 or 1");
  c.vec(vec_handle);
  (which == 0 ? c.oper(h).aux0 : c.oper(h).aux1) = vec_handle;
  API_END
}
pnp_status pnp_operator_set_valency(pnp_ctx* ctx, int h, double valency) { API_BEGIN(ctx) c.oper(h).valency = valency; API_END }
pnp_status pnp_constraints_get(pnp_ctx* ctx, int h, char* out) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.constraints_built, PNP_E_ARG, "constraints not built");
  const Operator& op = c.oper(h);
  if (c.degree >= 2) { p2_constraints_get(c, op, out); return PNP_OK; }
  const int F = op_fields(op.op);
  std::vector<unsigned char> m = c.dmask.to_host(c.stream);
  std::vector<int> i2e = c.int2ext.to_host(c.stream);
  for (long v = 0; v < c.nv; v++)
    for (int k = 0; k < F; k++) out[(long)k * c.nv + i2e[v]] = (char)((m[v] >> (F == 3 ? k : op.comp0)) & 1);
  API_END
}
pnp_status pnp_pattern_get(pnp_ctx* ctx, int h, long* nnz, int* rowptr, int* col) {
  API_BEGIN(ctx)
  long n = pattern_export(c, h, rowptr, col);
  if (nnz) *nnz = n;
  API_END
}

pnp_status pnp_vec_create(pnp_ctx* ctx, int fields, int* handle) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.finalized, PNP_E_ARG, "mesh not finalized");
  PNP_REQUIRE((fields == 1 || fields == 3) && handle, PNP_E_ARG, "fields must be 1 or 3");
  auto v = std::make_unique<Vec>();
  v->fields = fields; v->d.alloc((size_t)fields * c.cols()); v->d.zero(c.stream);
  c.vecs.push_back(std::move(v));
  *handle = (int)c.vecs.size() - 1;
  API_END
}
pnp_status pnp_vec_destroy(pnp_ctx* ctx, int h) {
  API_BEGIN(ctx)
  // a multigrid set up later must not re-discretise at a state that no longer exists
  if (c.vec(h).d.p == c.last_u) { c.last_u = nullptr; c.last_vals = nullptr; }
  c.vecs[h].reset();
  API_END
}
pnp_status pnp_vec_upload(pnp_ctx* ctx, int h, const double* host) { API_BEGIN(ctx) vec_upload(c, c.vec(h), host); API_END }
pnp_status pnp_vec_download(pnp_ctx* ctx, int h, double* host) { API_BEGIN(ctx) vec_download(c, c.vec(h), host); API_END }
pnp_status pnp_vec_set(pnp_ctx* ctx, int h, double value) {
  API_BEGIN(ctx)
  Vec& v = c.vec(h);
  k_fill<<<grid_for((long)v.d.n, 256), 256, 0, c.stream>>>(v.d.p, (long)v.d.n, value);
  PNP_CHECK_LAUNCH(); c.launches++;
  API_END
}
pnp_status pnp_vec_copy(pnp_ctx* ctx, int dst, int src) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.vec(dst).d.n == c.vec(src).d.n, PNP_E_ARG, "vector sizes differ");
  vec_copy(c, c.vec(src).d.p, c.vec(dst).d.p, (long)c.vec(src).d.n);
  API_END
}
pnp_status pnp_vec_axpy(pnp_ctx* ctx, int y, double a, int x) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.vec(y).d.n == c.vec(x).d.n, PNP_E_ARG, "vector sizes differ");
  vec_axpy(c, a, c.vec(x).d.p, c.vec(y).d.p, (long)c.vec(x).d.n);
  API_END
}
pnp_status pnp_vec_norm(pnp_ctx* ctx, int x, double* out) {
  API_BEGIN(ctx) *out = vec_norm(c, c.vec(x).d.p, c.rows() * c.vec(x).fields); API_END
}
pnp_status pnp_vec_dot(pnp_ctx* ctx, int x, int y, double* out) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.vec(y).d.n == c.vec(x).d.n, PNP_E_ARG, "vector sizes differ");
  *out = vec_dot(c, c.vec(x).d.p, c.vec(y).d.p, c.rows() * c.vec(x).fields);
  API_END
}
pnp_status pnp_vec_pack3(pnp_ctx* ctx, int dst3, int phi, int cp, int cm) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.vec(dst3).fields == 3 && c.vec(phi).fields == 1 && c.vec(cp).fields == 1 && c.vec(cm).fields == 1,
              PNP_E_ARG, "pack3 needs one 3-field and three 1-field vectors");
  if (c.degree >= 2) { // field-lexicographic layout: three block copies
    const int src[3] = {phi, cp, cm};
    for (int k = 0; k < 3; k++) vec_copy(c, c.vec(src[k]).d.p, c.vec(dst3).d.p + k * c.p2_nd, c.p2_nd);
    return PNP_OK;
  }
  k_pack3<<<grid_for(c.nv, 256), 256, 0, c.stream>>>(c.vec(phi).d.p, c.vec(cp).d.p, c.vec(cm).d.p, c.nv, c.vec(dst3).d.p);
  PNP_CHECK_LAUNCH(); c.launches++;
  API_END
}
pnp_status pnp_vec_extract(pnp_ctx* ctx, int src3, int field, int dst1) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.vec(src3).fields == 3 && c.vec(dst1).fields == 1 && field >= 0 && field < 3, PNP_E_ARG, "bad extract arguments");
  if (c.degree >= 2) { vec_copy(c, c.vec(src3).d.p + field * c.p2_nd, c.vec(dst1).d.p, c.p2_nd); return PNP_OK; }
  k_extract<<<grid_for(c.nv, 256), 256, 0, c.stream>>>(c.vec(src3).d.p, c.nv, field, c.vec(dst1).d.p);
  PNP_CHECK_LAUNCH(); c.launches++;
  API_END
}

pnp_status pnp_matrix_create(pnp_ctx* ctx, int op_handle, int* handle) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.finalized && handle, PNP_E_ARG, "mesh not finalized");
  auto m = std::make_unique<Matrix>();
  m->op = c.oper(op_handle).op; m->nplanes = op_planes(m->op);
  if (m->op == OP_PNP && tune().matrix_compact) m->nplanes = pnp_context_planes(c, JAC_ANALYTIC, true);
  if (c.degree >= 2) { PNP_REQUIRE(c.constraints_built, PNP_E_ARG, "constraints not built"); p2_matrix_init(c, *m, c.oper(op_handle)); }
  else { m->vals.alloc((size_t)m->nplanes * c.nslots); m->vals.zero(c.stream); }
  c.mats.push_back(std::move(m));
  *handle = (int)c.mats.size() - 1;
  API_END
}
pnp_status pnp_matrix_destroy(pnp_ctx* ctx, int h) {
  API_BEGIN(ctx)
  if (c.mat(h).vals.p == c.last_vals) c.last_vals = nullptr;
  c.mats[h].reset();
  API_END
}
pnp_status pnp_residual(pnp_ctx* ctx, int op, int u, int r) {
  API_BEGIN(ctx)
  assemble_residual(c, c.oper(op), c.vec(u), c.vec(r));
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}
pnp_status pnp_jacobian(pnp_ctx* ctx, int op, int u, int A, int mode, double eps) {
  API_BEGIN(ctx)
  assemble_jacobian(c, c.oper(op), c.vec(u), c.mat(A), mode, eps);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}
pnp_status pnp_matrix_values_get(pnp_ctx* ctx, int op, int A, double* val) {
  API_BEGIN(ctx) matrix_export(c, op, c.mat(A), val); API_END
}
pnp_status pnp_spmv(pnp_ctx* ctx, int A, int x, int y) {
  API_BEGIN(ctx)
  const Matrix& M = c.mat(A);
  PNP_REQUIRE(c.vec(x).fields == (M.nplanes == 1 ? 1 : 3) && c.vec(y).fields == c.vec(x).fields && x != y, PNP_E_ARG,
              "spmv operands do not match the matrix");
  spmv(c, M, c.vec(x).d.p, c.vec(y).d.p);
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}

pnp_status pnp_solver_create(pnp_ctx* ctx, int kind, int prec, int maxit, int prec_steps, int verbosity, int* handle) {
  API_BEGIN(ctx)
  PNP_REQUIRE((kind == PNP_SOLVER_BCGS || kind == PNP_SOLVER_CG) && prec >= PNP_PREC_NONE && prec <= PNP_PREC_AMG && handle,
              PNP_E_ARG, "bad solver arguments");
  auto s = std::make_unique<Solver>();
  s->kind = kind; s->prec = prec; s->maxit = maxit; s->prec_steps = prec_steps; s->verbosity = verbosity;
  c.solvers.push_back(std::move(s));
  *handle = (int)c.solvers.size() - 1;
  API_END
}
pnp_status pnp_solver_set_option(pnp_ctx* ctx, int s, const char* name, double value) {
  API_BEGIN(ctx)
  PNP_REQUIRE(name, PNP_E_ARG, "null option name");
  c.solver(s).opts[name] = value;
  API_END
}
pnp_status pnp_solver_get(pnp_ctx* ctx, int s, const char* name, double* value) {
  API_BEGIN(ctx)
  PNP_REQUIRE(name && value, PNP_E_ARG, "null argument");
  const std::string n(name);
  if (c.degree >= 2 && (n == "ssor_levels" || n == "ilu0_levels")) *value = c.solver(s).csr_levels;
  else if (n == "ssor_levels") *value = sweep_levels(c.solver(s), false);
  else if (n == "ilu0_levels") *value = sweep_levels(c.solver(s), true);
  else if (n == "amg_graph") *value = amg_graph_state(c.solver(s));
  else PNP_REQUIRE(false, PNP_E_ARG, "unknown solver fact");
  API_END
}
pnp_status pnp_precond_apply(pnp_ctx* ctx, int s, int A, int d, int v) {
  API_BEGIN(ctx)
  precond_apply(c, c.solver(s), c.mat(A), c.vec(d), c.vec(v));
  PNP_CUDA(cudaStreamSynchronize(c.stream));
  API_END
}
pnp_status pnp_solver_apply(pnp_ctx* ctx, int s, int A, int z, int r, double reduction, pnp_lin_result* out) {
  API_BEGIN(ctx)
  LinResult lr = solver_apply(c, c.solver(s), c.mat(A), c.vec(z), c.vec(r), reduction);
  to_lin(lr, out);
  if (lr.status == PNP_E_BREAKDOWN) { c.err = "BiCGSTAB breakdown (rho, omega or h vanished)"; return PNP_E_BREAKDOWN; }
  if (lr.status == PNP_E_NAN) { c.err = "non-finite residual norm in the linear solver"; return PNP_E_NAN; }
  API_END
}

void pnp_newton_opts_default(pnp_newton_opts* o) {
  if (!o) return;
  // PDELab Newton defaults (SURVEY App. A.1)
  o->reduction = 1e-8; o->abs_limit = 1e-12; o->min_linear_reduction = 1e-3; o->reassemble_threshold = 0.0;
  o->max_iterations = 40; o->line_search_max_iterations = 10; o->damping = 0.5;
  o->jac_mode = PNP_JAC_FD_FAITHFUL; o->fd_epsilon = 1e-11; o->verbosity = 0;
  o->line_search_strategy = PNP_LS_HACKBUSCH_REUSKEN_ACCEPT_BEST;
}
pnp_status pnp_newton_opts_from_params(pnp_ctx* ctx, pnp_newton_opts* o) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.params.set && o, PNP_E_ARG, "parameters not set");
  pnp_newton_opts_default(o);
  o->reassemble_threshold = c.params.newtonReassembleThreshold;
  o->reduction = c.params.newtonReduction;
  o->min_linear_reduction = c.params.newtonMinLinearReduction;
  o->max_iterations = (int)c.params.newtonMaxIterations;                       // stored as double (quirk B10)
  o->line_search_max_iterations = (int)c.params.newtonLineSearchMaxIteration;
  o->verbosity = c.params.verbosity;
  API_END
}
pnp_status pnp_newton_apply(pnp_ctx* ctx, int op, int u, int solver, const pnp_newton_opts* o, pnp_newton_result* res) {
  API_BEGIN(ctx)
  PNP_REQUIRE(o && res, PNP_E_ARG, "null options/result");
  int st = newton_apply(c, c.oper(op), c.vec(u), c.solver(solver), *o, *res);
  if (st != PNP_OK) {
    static const char* msg[] = {"", "Newton did not converge within max_iterations", "linear solver did not converge",
                                "line search failed", "defect is not finite", "BiCGSTAB breakdown"};
    c.err = msg[st <= 5 ? st : 0];
    return st;
  }
  API_END
}
pnp_status pnp_slp_apply(pnp_ctx* ctx, int op, int u, int solver, double reduction, int jac_mode, double eps,
                         pnp_lin_result* out) {
  API_BEGIN(ctx)
  LinResult lr = slp_apply(c, c.oper(op), c.vec(u), c.solver(solver), reduction, jac_mode, eps);
  to_lin(lr, out);
  if (lr.status == PNP_E_BREAKDOWN) { c.err = "BiCGSTAB breakdown (rho, omega or h vanished)"; return PNP_E_BREAKDOWN; }
  if (lr.status == PNP_E_NAN) { c.err = "non-finite residual norm in the linear solver"; return PNP_E_NAN; }
  API_END
}
pnp_status pnp_onestep_apply(pnp_ctx* ctx, int method, int op_space, int op_time, int solver, double time, double dt,
                             int x_old, int dirichlet_values, int x_new, double reduction, int jac_mode, double eps,
                             pnp_lin_result* stage_results) {
  API_BEGIN(ctx)
  (void)time; // the reference's boundary functions and operators do not depend on time
  LinResult lr[2];
  const int st = onestep_apply(c, method, c.oper(op_space), c.oper(op_time), c.solver(solver), dt, c.vec(x_old),
                               c.vec(dirichlet_values), c.vec(x_new), reduction, jac_mode, eps, lr);
  if (stage_results) for (int k = 0; k < (method == PNP_TIME_IMPLICIT_EULER ? 1 : 2); k++) to_lin(lr[k], stage_results + k);
  if (st == PNP_E_BREAKDOWN) { c.err = "BiCGSTAB breakdown in a stage solve"; return PNP_E_BREAKDOWN; }
  if (st == PNP_E_NAN) { c.err = "non-finite residual norm in a stage solve"; return PNP_E_NAN; }
  API_END
}
pnp_status pnp_ion_flux(pnp_ctx* ctx, int phi, int cp, int cm, double* ip, double* im) {
  API_BEGIN(ctx)
  PNP_REQUIRE(ip && im, PNP_E_ARG, "null output");
  ion_flux(c, c.vec(phi), c.vec(cp), c.vec(cm), ip, im);
  API_END
}
pnp_status pnp_write_cell_data(pnp_ctx* ctx, int v, const char* filename) {
  API_BEGIN(ctx)
  PNP_REQUIRE(filename, PNP_E_ARG, "null file name");
  write_cell_data(c, c.vec(v), filename);
  API_END
}
pnp_status pnp_write_vtk(pnp_ctx* ctx, const char* name, int n, const int* vec_handles, const char* const* names, int ascii) {
  API_BEGIN(ctx)
  PNP_REQUIRE(name && n >= 0 && (n == 0 || (vec_handles && names)), PNP_E_ARG, "null arguments");
  std::vector<const Vec*> f(n);
  for (int i = 0; i < n; i++) f[i] = &c.vec(vec_handles[i]);
  write_vtk(c, name, n, f.data(), names, ascii);
  API_END
}
pnp_status pnp_matrix_set_csr(pnp_ctx* ctx, int op_handle, int mat_handle, const int* rowptr, const int* col, const double* val) {
  API_BEGIN(ctx) matrix_import(c, op_handle, c.mat(mat_handle), rowptr, col, val); API_END
}
pnp_status pnp_mesh_renumber(pnp_ctx* ctx, const int* new_index) { API_BEGIN(ctx) mesh_renumber(c, new_index); API_END }
pnp_status pnp_mesh_owned(pnp_ctx* ctx, long* n_own) { API_BEGIN(ctx) if (n_own) *n_own = c.n_own; API_END }
pnp_status pnp_interpolate_bcext(pnp_ctx* ctx, int component, int pb_vec, int out_vec) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.n_own == c.nv, PNP_E_ARG, "interpolate(BCExtension) follows the global element order: run it before partitioning");
  if (c.degree >= 2) p2_interpolate_bcext(c, component, pb_vec >= 0 ? &c.vec(pb_vec) : nullptr, c.vec(out_vec));
  else interpolate_bcext(c, component, pb_vec >= 0 ? &c.vec(pb_vec) : nullptr, c.vec(out_vec));
  API_END
}
// ---- quadratic elements (-DPDEGREE=2 builds of the reference, src/Makefile.am:57-110) ----
pnp_status pnp_space_set_degree(pnp_ctx* ctx, int degree) {
  API_BEGIN(ctx)
  PNP_REQUIRE(degree >= 1 && degree <= 3, PNP_E_ARG, "polynomial degree must be 1, 2 or 3");
  PNP_REQUIRE(!c.finalized, PNP_E_ARG, "set the degree before pnp_mesh_finalize");
  PNP_REQUIRE(degree == 1 || (c.world == 1 && !c.parent), PNP_E_ARG, "quadratic and cubic elements run on one GPU");
  c.degree = degree;
  API_END
}
pnp_status pnp_space_sizes(pnp_ctx* ctx, int* degree, long* n_edges, long* ndof) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.finalized, PNP_E_ARG, "mesh not finalized");
  if (degree) *degree = c.degree;
  if (c.degree >= 2) p2_sizes(c, n_edges, ndof);
  else { if (n_edges) *n_edges = 0; if (ndof) *ndof = c.nv; }
  API_END
}
pnp_status pnp_space_edges(pnp_ctx* ctx, int* va, int* vb) { API_BEGIN(ctx) p2_edges(c, va, vb); API_END }
pnp_status pnp_space_offsets(pnp_ctx* ctx, long* edge_offset, long* vertex_offset) {
  API_BEGIN(ctx)
  PNP_REQUIRE(c.finalized, PNP_E_ARG, "mesh not finalized");
  if (c.degree >= 2) p2_offsets(c, edge_offset, vertex_offset);
  else { if (edge_offset) *edge_offset = 0; if (vertex_offset) *vertex_offset = 0; }
  API_END
}
pnp_status pnp_operator_set_intorder(pnp_ctx* ctx, int h, int intorder) {
  API_BEGIN(ctx)
  PNP_REQUIRE(intorder == 0 || (intorder == 5 && c.degree >= 2), PNP_E_ARG,
              "quadrature order: 0 (the order the reference's drivers end up with) or, for degree 2 and 3, 5");
  c.oper(h).intorder = intorder;
  API_END
}

} // extern "C"
