// pnp_common.cuh -- context, device buffers, error handling shared by the .cu translation units.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/pnp_b200.h"
#include "pnp_setup_algos.cuh"
#include "pnp_star.cuh"

namespace pnp {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define PNP_CUDA(call)                                                                               \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess)                                                                           \
      throw ::pnp::Error(PNP_E_CUDA, std::string(__FILE__) + ":" + std::to_string(__LINE__) + " " +  \
                                         #call + " -> " + cudaGetErrorString(e_));                   \
  } while (0)
#define PNP_CHECK_LAUNCH() PNP_CUDA(cudaGetLastError())
#define PNP_REQUIRE(cond, code, msg)                                                                 \
  do { if (!(cond)) throw ::pnp::Error(code, std::string(msg)); } while (0)

// Plain owning device array.
template <class T> struct DBuf {
  T* p = nullptr;
  size_t n = 0;
  DBuf() = default;
  explicit DBuf(size_t n_) { alloc(n_); }
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  DBuf(DBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DBuf& operator=(DBuf&& o) noexcept { if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; } return *this; }
  ~DBuf() { release(); }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
  // 64 bytes of slack behind every array: the bulk copies of the streaming kernels (pnp_spmv_tma.cuh) round their
  // extent up to 16 bytes and may read a few bytes past the last element
  void alloc(size_t n_) {
    release();
    n = n_;
    if (n) PNP_CUDA(cudaMalloc(&p, n * sizeof(T) + 64));
  }
  void zero(cudaStream_t s) { if (n) PNP_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
  void upload(const T* h, size_t cnt, cudaStream_t s) {
    if (cnt) PNP_CUDA(cudaMemcpyAsync(p, h, cnt * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  void download(T* h, size_t cnt, cudaStream_t s) const {
    if (cnt) PNP_CUDA(cudaMemcpyAsync(h, p, cnt * sizeof(T), cudaMemcpyDeviceToHost, s));
    PNP_CUDA(cudaStreamSynchronize(s));
  }
  std::vector<T> to_host(cudaStream_t s) const { std::vector<T> h(n); download(h.data(), n, s); return h; }
};

// process-wide tuning knobs (pnp_tune): experiments and tests switch kernel variants without rebuilding
struct Tune {
  int tma = 1;            // streaming (bulk-copy) SpMV for large levels; 0: plain-load kernel everywhere
  int tma_stages = 2;     // ring depth of the streaming SpMV (2..3); two stages leave more of the SM's memory to L1
  int tma_lpr = 2;        // lanes per row in the streaming SpMV (1 or 2): 2 -> eight consumer warps per SM
  long tma_min_rows = -1; // smallest level the streaming SpMV serves (-1: two tiles per SM)
  int graph = 1;          // the multigrid's coarse correction is replayed from a CUDA graph
  int fd_warp = 1;        // FD-faithful Jacobian: warp-cooperative kernel (0: one thread per vertex)
  int jac_compact = 1;    // Newton / linear-problem Jacobian in the compact 5-plane PNP layout where it applies (0: always 7)
  int matrix_compact = 0; // pnp_matrix_create: PNP matrices in the compact layout where the exact Jacobian has it (0: always 7)
  long p2_chunk = 0;      // quadratic / cubic elements: elements per scratch block of the Jacobian assembly (0: 2 GB worth)
};
inline Tune& tune() { static Tune t; return t; }

inline int grid_for(long n, int block, int max_blocks = 148 * 32) {
  long g = (n + block - 1) / block;
  if (g < 1) g = 1;
  return (int)(g > max_blocks ? max_blocks : g);
}

// ---- host-side parameter set (Sysparams / Surface of the reference, sysparams.hh:10-57) ----
struct HostSurface { int btype[3] = {1, 1, 1}; double flux[3] = {0, 0, 0}; double dval[3] = {0, 0, 0}; };
struct HostParams {
  bool set = false;
  int n_surfaces = 0, verbosity = 0, cylindrical = 0;
  double l_b = 1, c0 = 0.06, PI = 3.1415;
  int linearSolverIterations = 50;
  double newtonReassembleThreshold = 0, newtonReduction = 1e-5, newtonMinLinearReduction = 1e-5;
  double newtonMaxIterations = 50, newtonLineSearchMaxIteration = 500, tau = 0.1;
  int nSteps = 100, outputFreq = 1, potentialUpdateFreq = 1;
  std::string meshfile;
  std::vector<HostSurface> surfaces;
};

struct Vec {
  int fields = 1;
  DBuf<double> d; // vertex-blocked internal layout, fields*nv
};
struct Matrix {
  int op = 0;
  int nplanes = 1;   // value planes: 1 (scalar operators), 7 (PNP, pnp_plane()) or 5 (compact PNP, pnp_block())
  int comp0 = 0;  // BC component of the operator that assembled it (scalar operators)
  DBuf<double> vals; // nplanes * nslots (star layout) or csr_nnz (quadratic elements)
  // quadratic elements (pnp_p2.cu): scalar CSR in the reference's dof numbering; the pattern belongs to the space
  const int* csr_rp = nullptr; const int* csr_col = nullptr; long csr_nnz = 0, csr_n = 0;
  void* csr_pattern = nullptr; // the P2Pattern the pointers belong to (level schedule of the sweeps)
};

struct Operator {
  int op = OP_PB;
  int comp0 = 0;          // BC component of a scalar operator's BCType
  double valency = 1.0;
  int aux0 = -1, aux1 = -1; // vector handles of coefficient fields
  int intorder = 0;         // quadrature order (degree 2 / 3 only): 0 = the reference drivers' (3; diffusion 2, mass 5), 5 = 7-point rule
};

// One coarser level of the refinement hierarchy, captured by mesh_refine(): that level's vertex star (own locality
// numbering) and the edges whose midpoints became the next finer level's new vertices (reference numbering of this
// level: vertex nv + k of the finer level is the midpoint of edge k).  Feeds the geometric levels of the multigrid
// preconditioner (pnp_amg.cu).
struct HierLevel {
  long nv = 0, nslots = 0, nE = 0;
  DBuf<int> rp, int2ext, ext2int;
  DBuf<unsigned> adj;
  DBuf<uint64_t> edges; // (min << 32 | max), sorted
};

struct Ctx;
// One coarser level of a DISTRIBUTED multigrid hierarchy: a child context holding this rank's part of the coarser mesh
// (own star, Dirichlet mask, halo plan) and, for every local vertex of the next finer level (internal numbering), its
// parents on this level (internal numbering, -1: none).
struct MgLevelRef {
  Ctx* lc = nullptr;
  DBuf<int> par0, par1;
};

struct Amg; // pnp_amg.cu
struct P2Space; // pnp_p2.cu
struct SweepPrec; // pnp_precond.cu: level schedules of the SSOR / ILU0 sweeps, ILU0 factor
struct SweepPlan; // pnp_precond.cu: one level schedule

struct Solver {
  int kind = PNP_SOLVER_BCGS, prec = PNP_PREC_NONE, maxit = 5000, prec_steps = 1, verbosity = 0;
  std::shared_ptr<Amg> amg;
  std::shared_ptr<SweepPrec> sweep;
  std::map<std::string, double> opts; // pnp_solver_set_option
  double opt(const char* name, double dflt) const { auto it = opts.find(name); return it == opts.end() ? dflt : it->second; }
  DBuf<double> w[6]; // Krylov work vectors, sized on first use
  DBuf<double> dinv; // Jacobi: inverse diagonal
  DBuf<double> csr_lu; int csr_levels = 0; // quadratic elements: ILU0 factor on the CSR pattern; levels of the last sweep set-up
  std::shared_ptr<void> pmg;               // quadratic / cubic elements: p-multigrid state (pnp_p2.cu)
  void ensure(size_t n) { for (auto& b : w) if (b.n != n) b.alloc(n); if (dinv.n != n) dinv.alloc(n); }
};

struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int sm_count = 148;
  // canonical mesh, device resident (external numbering = Gmsh-compressed / refinement rule)
  long nv = 0, nT = 0, nB = 0;
  // Rows exist for the first n_own vertices; on one GPU n_own == nv.  With a partitioned mesh the vertices
  // [n_own, nv) are ghosts: columns of owned rows whose values arrive by halo exchange (pnp_comm.cu).
  long n_own = 0;
  // polynomial degree of the finite element space (PDEGREE of the reference's build): 1 = vertex-star layout, 2 = the
  // edge + vertex dofs of pnp_p2.cu (p2_nd of them per field; vectors field-lexicographic, matrices CSR)
  int degree = 1; long p2_nd = 0;
  std::shared_ptr<P2Space> p2;
  long rows() const { return degree >= 2 ? p2_nd : n_own; } // dofs per field this rank owns
  long cols() const { return degree >= 2 ? p2_nd : nv; }    // ... and holds (owned + ghosts)
  int rank = 0, world = 1;
  void* nccl = nullptr;                 // ncclComm_t
  std::vector<int> halo_nbr, halo_send_ptr, halo_recv_ptr; // per neighbour rank: ranges into send list / ghost block
  std::vector<int> halo_send_ext;       // send list in the caller's local numbering
  DBuf<int> halo_send_idx;              // ... in internal numbering
  DBuf<double> halo_send_buf;
  DBuf<double> cx, cy;
  DBuf<int> ctri, cba, cbb, cbphys;
  // star structure, internal numbering
  bool finalized = false;
  long nslots = 0;
  DBuf<int> rp;
  DBuf<unsigned> adj;
  DBuf<XY> xy;
  DBuf<unsigned char> dmask;
  DBuf<int> int2ext, ext2int;
  // boundary
  std::vector<BFace> bfaces;           // host copy (O(sqrt N))
  DBuf<BFace> d_bfaces;
  DBuf<int> d_bv, d_bv_ptr, d_bv_items; // boundary-vertex incidence lists (vertex, ptr, face*4+role)
  int n_bv = 0;
  DBuf<double> d_surf;                 // per surface: flux[3]
  DBuf<unsigned char> d_surf_dir;      // per surface: bit c = component c is Dirichlet there
  HostParams params;
  bool constraints_built = false;
  long launches = 0;                   // kernels launched (bench.py reports gpu_launches)
  // ALGORITHMIC bytes moved since the last reset, by kernel class (bench.py's roofline.step): compulsory traffic of every
  // launch -- each array a kernel must read or write counted once (DESIGN.md section 3 lists the per-kernel figures)
  enum { ACC_SPMV_FINE = 0, ACC_SPMV_COARSE = 1, ACC_ASSEMBLY = 2, ACC_BLAS1 = 3, ACC_TRANSFER = 4, ACC_DENSE = 5, ACC_N = 6 };
  double alg_bytes[ACC_N] = {0, 0, 0, 0, 0, 0};
  void acct(int cls, double bytes) { alg_bytes[cls] += bytes; }
  // a level context's (child's) launches and bytes are the parent's
  void absorb(Ctx& child) {
    launches += child.launches; child.launches = 0;
    for (int k = 0; k < ACC_N; k++) { alg_bytes[k] += child.alg_bytes[k]; child.alg_bytes[k] = 0; }
  }
  // optional CUDA-event profile of the fine-level SpMV launches (bench.py's roofline leg)
  bool prof = false;
  std::vector<cudaEvent_t> prof_ev;
  std::vector<int> prof_kind;          // per event pair: 0 plain/dot SpMV, 1 residual epilogue, 2 smoother epilogue
  size_t prof_used = 0;
  cudaEvent_t tm0 = nullptr, tm1 = nullptr; // pnp_timer_start/stop
  void prof_mark(int kind = 0) {
    if (!prof) return;
    if (prof_used == prof_ev.size()) { cudaEvent_t e; cudaEventCreate(&e); prof_ev.push_back(e); }
    if (prof_used % 2 == 0) { if (prof_kind.size() <= prof_used / 2) prof_kind.resize(prof_used / 2 + 1); prof_kind[prof_used / 2] = kind; }
    cudaEventRecord(prof_ev[prof_used++], stream);
  }
  // handle tables
  std::vector<std::unique_ptr<Vec>> vecs;
  std::vector<std::unique_ptr<Matrix>> mats;
  std::vector<std::unique_ptr<Operator>> ops;
  std::vector<std::unique_ptr<Solver>> solvers;
  // Newton / SLP work space (r, z, previous iterate, Jacobian), kept between calls: allocating and freeing ~20 GB per
  // Newton call costs more than the step itself
  Vec ws_r, ws_z, ws_prev;
  Matrix ws_A;
  Vec ws_stage[6];                     // one-step method: stage vectors, constant residual part, operator residuals
  Matrix ws_B;                         // one-step method: Jacobian of the temporal operator
  DBuf<double> io_stage;               // vec_upload / vec_download: device staging in the reference's layout
  bool owns_stream = true;             // child contexts (coarser multigrid levels) share the parent's stream and communicator
  std::vector<MgLevelRef> mg;          // distributed multigrid: coarser levels, finest-but-one first
  // coarsest distributed level: internal vertex -> index in the replicated dense system.  mg_aggregated = false: that
  // index is the global vertex (the level itself is solved densely); true: it is an aggregate of global vertices (the
  // level is smoothed like the others and the Galerkin aggregate system below it is the dense one)
  DBuf<int> mg_gid; long mg_nglobal = 0; bool mg_aggregated = false;
  Ctx* mg_replica = nullptr;           // whole coarsest mesh on every rank: single-GPU multigrid below it (mg_gid maps into ITS internal numbering)
  long mg_epoch = 0;                   // bumped by every pnp_mg_* call: a multigrid built for an older hierarchy is rebuilt
  Ctx* parent = nullptr;               // child contexts: the context whose stream / communicator they borrow
  std::vector<Ctx*> children;          // ... and the children a context has handed out (their lifetime is bounded by the parent's)
  std::vector<void*> owned_children;   // pnp_ctx handles pnp_partition_build created: destroyed with this context
  bool owns_comm = false;
  // what the last assemble_jacobian() call linearised (coarse levels of the distributed multigrid re-discretise it)
  const double* last_u = nullptr; Operator last_op; int last_mode = 0; double last_eps = 1e-11;
  const double* last_vals = nullptr;   // ... and the matrix values it wrote (reset when they are combined into something else)
  std::vector<HierLevel> hier;         // coarser refinement levels, coarsest first
  std::vector<Vec> carry;              // nodal fields in reference numbering, interpolated by mesh_refine()
  // a new / refined mesh invalidates every object sized by it
  void invalidate_mesh_objects() {
    finalized = false; constraints_built = false; p2.reset(); p2_nd = 0;
    vecs.clear(); mats.clear(); ops.clear(); solvers.clear();
    last_u = nullptr; last_vals = nullptr;
    ws_r.d.release(); ws_z.d.release(); ws_prev.d.release(); ws_A.vals.release(); ws_B.vals.release();
    for (auto& v : ws_stage) v.d.release();
    io_stage.release();
  }
  // scratch for reductions
  DBuf<double> red_partial, red_out;
  double* h_red = nullptr; // pinned

  StarView star() const { return StarView{rp.p, adj.p, xy.p, dmask.p, (int)n_own}; }
  PhysParams phys(double valency) const {
    PhysParams P; P.PI = params.PI; P.l_b = params.l_b; P.c0 = params.c0; P.valency = valency;
    P.cylindrical = params.cylindrical; return P;
  }
  Vec& vec(int h) { PNP_REQUIRE(h >= 0 && h < (int)vecs.size() && vecs[h], PNP_E_ARG, "bad vector handle"); return *vecs[h]; }
  Matrix& mat(int h) { PNP_REQUIRE(h >= 0 && h < (int)mats.size() && mats[h], PNP_E_ARG, "bad matrix handle"); return *mats[h]; }
  Operator& oper(int h) { PNP_REQUIRE(h >= 0 && h < (int)ops.size() && ops[h], PNP_E_ARG, "bad operator handle"); return *ops[h]; }
  Solver& solver(int h) { PNP_REQUIRE(h >= 0 && h < (int)solvers.size() && solvers[h], PNP_E_ARG, "bad solver handle"); return *solvers[h]; }
};

inline int op_fields(int op) { return op == OP_PNP ? 3 : 1; }
inline int op_planes(int op) { return op == OP_PNP ? 7 : 1; }

// ---- implemented across the translation units ----
// pnp_setup.cu
void mesh_set(Ctx&, long nv, const double* x, const double* y, long nT, const int* tri, long nB, const int* ba,
              const int* bb, const int* bphys, long n_own);
void mesh_refine(Ctx&, int levels);
void mesh_finalize(Ctx&, bool renumber);
void constraints_build(Ctx&);
// pnp_comm.cu
void comm_init(Ctx&, int rank, int world, const char* unique_id128);
void comm_unique_id(char* out128);
void comm_destroy(Ctx&);
void comm_bootstrap_file(Ctx&, int rank, int world, const std::string& path);
std::vector<unsigned char> comm_allgatherv(Ctx&, const void* send, long nbytes, std::vector<long>& counts);
void halo_set(Ctx&, int n_nbr, const int* nbr, const int* send_ptr, const int* send_idx, const int* recv_ptr);
void halo_finalize(Ctx&);
void halo_exchange(Ctx&, double* x, int fields);
void allreduce_sum(Ctx&, double* dev, size_t n);
void allreduce_max_u64(Ctx&, unsigned long long* dev, size_t n);
void carry_set(Ctx&, const int* handles, int n);
void carry_get(Ctx&, int i, Vec& out);
void vec_upload(Ctx&, Vec&, const double* host_lex);
void vec_download(Ctx&, const Vec&, double* host_lex);
void vec_from_lex_device(Ctx&, Vec&, const double* d_lex);
void vec_to_lex_device(Ctx&, const Vec&, double* d_lex);
Ctx* ctx_make_owned_child(Ctx& parent); // pnp_capi.cu: a context on the parent's stream, destroyed with the parent ...
void ctx_destroy_owned_child(Ctx& parent, Ctx* child); // ... or earlier
long pattern_export(Ctx&, int op_handle, int* rowptr, int* col);
void matrix_export(Ctx&, int op_handle, const Matrix&, double* val);
void matrix_import(Ctx&, int op_handle, Matrix&, const int* rowptr, const int* col, const double* val);
void mesh_renumber(Ctx&, const int* new_index);
// pnp_host.cpp-like logic in pnp_hostside.cu
void read_gmsh_file(const std::string& path, std::vector<double>& x, std::vector<double>& y, std::vector<int>& tri,
                    std::vector<int>& ba, std::vector<int>& bb, std::vector<int>& bphys);
void read_config_file(const std::string& path, HostParams& p);
void interpolate_bcext(Ctx&, int comp, const Vec* pb, Vec& out);
// pnp_assembly.cu
void assemble_residual(Ctx&, const Operator&, Vec& u, Vec& r);   // refreshes the ghost part of u
void assemble_jacobian(Ctx&, const Operator&, Vec& u, Matrix& A, int mode, double eps);
void assemble_jacobian_on(Ctx&, const StarView& M, long stride, const Operator&, const double* u, double* vals, int nplanes,
                          int mode, double eps);
// pnp_linalg.cu
void spmv(Ctx&, const Matrix& A, double* x, double* y); // refreshes the ghost part of x
double vec_norm(Ctx&, const double* x, long n);
double vec_dot(Ctx&, const double* x, const double* y, long n);
void vec_axpy(Ctx&, double a, const double* x, double* y, long n);
void vec_copy(Ctx&, const double* x, double* y, long n);
void vec_zero(Ctx&, double* x, long n);
struct LinResult { bool converged = false; int iterations = 0; double reduction = 1, conv_rate = 1; int status = 0; double seconds = 0; };
LinResult solver_apply(Ctx&, Solver&, const Matrix& A, Vec& z, Vec& r, double reduction);
void precond_apply(Ctx&, Solver&, const Matrix& A, Vec& d, Vec& v); // v = M^-1 d (setup + one application)
// pnp_precond.cu
int sweep_levels(const Solver&, bool ilu);
// pnp_p2.cu (quadratic elements)
void p2_build(Ctx&);
void p2_constraints(Ctx&);
void p2_matrix_init(Ctx&, Matrix&, const Operator&);
void p2_assemble_residual(Ctx&, const Operator&, Vec& u, Vec& r);
void p2_assemble_jacobian(Ctx&, const Operator&, Vec& u, Matrix& A, int mode, double eps);
void csr_spmv(Ctx&, const Matrix& A, const double* x, double* y);
void csr_diag_inverse(Ctx&, const Matrix& A, double* dinv);
void csr_sweep_setup(Ctx&, Solver&, const Matrix& A, bool ilu);
void csr_ssor_apply(Ctx&, Solver&, const Matrix& A, const double* d, double* y);
void csr_ilu0_apply(Ctx&, Solver&, const Matrix& A, const double* d, double* y);
void pmg_setup(Ctx&, Solver&, const Matrix& A);
void pmg_apply(Ctx&, Solver&, const Matrix& A, const double* d, double* y);
const unsigned char* p2_dirichlet_flags(Ctx&); // per scalar dof: bit c = Dirichlet for BC component c (device)
void p2_sizes(Ctx&, long* nE, long* nd);
void p2_offsets(Ctx&, long* eoff, long* voff);
void p2_edges(Ctx&, int* eva, int* evb);
void p2_constraints_get(Ctx&, const Operator&, char* out);
long p2_pattern_export(Ctx&, const Operator&, int* rowptr, int* col);
void p2_matrix_import(Ctx&, const Operator&, Matrix&, const int* rowptr, const int* col, const double* val);
void p2_interpolate_bcext(Ctx&, int comp, const Vec* pb, Vec& out);
void p2_ion_flux(Ctx&, const Vec& phi, const Vec& cp, const Vec& cm, double* ip, double* im);
void p2_write_cell_data(Ctx&, const Vec& u, const std::string& filename);
void p2_vertex_values(Ctx&, const Vec& u, double* out);
// pnp_output.cu
void ion_flux(Ctx&, const Vec& phi, const Vec& cp, const Vec& cm, double* ip, double* im);
void write_cell_data(Ctx&, const Vec& u, const std::string& filename);
void write_vtk(Ctx&, const std::string& name, int nfields, const Vec* const* fields, const char* const* names, int ascii);

} // namespace pnp

// the opaque handle of the C ABI
struct pnp_ctx { pnp::Ctx c; };
