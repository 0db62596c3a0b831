// Handle definitions behind the opaque hdd_mesh / hdd_swipdg pointers.
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "common.hpp"
#include "kernels.hpp"

struct ncclComm;

namespace hdd {

// thin, lazily dlopen'ed NCCL binding (libnccl.so.2 - the copy torch already loaded, if any)
struct Nccl {
  static Nccl& get();
  bool available() const { return handle_ != nullptr; }
  void unique_id(void* id128);
  ncclComm* init_rank(const void* id128, int rank, int world);
  void destroy(ncclComm* c);
  void all_reduce_sum(double* buf, size_t count, ncclComm* c, cudaStream_t s);
  void all_reduce_min(double* buf, size_t count, ncclComm* c, cudaStream_t s);
  void all_gather_bytes(const void* send, void* recv, size_t bytes_per_rank, ncclComm* c, cudaStream_t s);
  void group_start();
  void group_end();
  void send(const double* buf, size_t count, int peer, ncclComm* c, cudaStream_t s);
  void recv(double* buf, size_t count, int peer, ncclComm* c, cudaStream_t s);

 private:
  Nccl();
  void check(int result, const char* what);
  void* handle_ = nullptr;
  void* fn_[12] = {};
};

struct HaloPeer {
  int rank;
  int64_t send_offset, send_count;  // in cells, into the list of cells to pack
  int64_t recv_offset, recv_count;  // in cells: a contiguous range of local cells (halo sorted by global id)
};

}  // namespace hdd

struct hdd_comm {
  int rank = 0, world = 1, device = 0;
  ncclComm* comm = nullptr;
};

struct hdd_mesh {
  int kind = 0, nl = 0, nf = 0, device = 0;
  cudaStream_t stream = nullptr;
  int64_t n_global = 0, cell_begin = 0, cell_end = 0;
  int32_t n_loc = 0, own0 = 0, n_own = 0;
  int32_t n_verts_loc = 0;

  // host copies needed after creation
  std::vector<int32_t> cgid;       // global ids of the halo cells, sorted (lower halo, then upper halo); empty for a whole mesh
  bool whole = true;               // this rank owns every cell
  // global id of a local cell: [lower halo | owned | upper halo]; `cgid` holds the halo cells only (sorted)
  int32_t gid(int32_t lc) const {
    if (whole) return lc;
    if (lc < own0) return cgid[size_t(lc)];
    if (lc < own0 + n_own) return int32_t(cell_begin) + (lc - own0);
    return cgid[size_t(lc - n_own)];
  }
  int n_subdomains = 1;
  std::vector<int64_t> sub_cell_offsets;             // [n_subdomains+1] global cell offsets
  std::vector<int64_t> sub_dof_offsets;              // nl * sub_cell_offsets
  std::vector<std::vector<int32_t>> sub_neighbours;  // [n_subdomains]
  std::vector<double> sub_diameter;                  // [n_subdomains], owned subdomains only (else 0)
  int sub_first = 0, sub_last = 0;                   // owned subdomains [sub_first, sub_last)
  std::vector<int64_t> seg_ptr;                      // chunked owned-cell segments for deterministic sums
  std::vector<int32_t> seg_sub;                      // subdomain of each segment

  // device
  hdd::DevBuf<double> cgeo;
  hdd::DevBuf<int32_t> neigh, d_cgid, cell_verts;
  hdd::DevBuf<uint8_t> btype, vboundary;
  hdd::DevBuf<int64_t> blk_start, vptr, d_seg_ptr;
  hdd::DevBuf<int32_t> vdof;
  int64_t n_blocks = 0;  // blk_start[n_own]
  bool has_btype = false;
  // logically structured cube grid (vertices x-fastest): cells per direction (0 = not structured / not one GPU), the
  // vertex 0 of every cell and the map lexicographic cell -> cell; feeds the multigrid preconditioner ("cg.mg")
  int sx = 0, sy = 0;
  // simplex grid whose vertices form a tensor-product lattice numbered x-fastest and whose triangles join lattice neighbours
  // (the ALU ladder of the test cases): lattice cells per direction, global (= lattice) vertex ids of the local cells and of
  // the local vertices - what cg.mg needs for its conforming P1 auxiliary space
  int lx = 0, ly = 0;
  hdd::DevBuf<int32_t> cell_gv, lvert_gid;
  hdd::DevBuf<int32_t> cell_v0, lex_cell;
  hdd::DevBuf<double> tgeo;  // {x0, hx, 1/hx, -} per column, {y0, hy, 1/hy, -} per row
  bool purely_neumann = false;  // no Dirichlet face anywhere (DirichletDetector, discretizations/swipdg.hh:219-220,488-489)

  // multi GPU
  int rank = 0, world = 1;
  ncclComm* comm = nullptr;
  std::vector<int64_t> rank_cell_offsets;  // [world+1]
  std::vector<hdd::HaloPeer> peers;
  hdd::DevBuf<int32_t> send_idx;  // local cells whose DoFs are packed, grouped by peer
  hdd::DevBuf<double> send_buf;
  int64_t n_send_cells = 0, send_buf_capacity = 0;
  hdd::DevBuf<int32_t> halo_peer, halo_rcell;  // per halo cell: owner rank, cell offset inside the owner's owned range
  std::vector<int32_t> rank_own0;              // own0 of every rank
  // host scratch used while the halo plan is built
  // for the halo plan of hdd_mesh_attach_comm (the caller's arrays are gone by then): global vertex ids of the halo cells
  // [n_halo*nl] (halo order), the owned cells along the partition boundary (local ids, sorted) and their vertex ids
  std::vector<int32_t> h_halo_verts, h_bowned, h_bowned_verts;
  int64_t v_begin = 0, v_end = 0;  // vertex id range the local cells touch

  hdd::MeshView view(const double* tensor) const {
    hdd::MeshView v{};
    v.kind = kind;
    v.nl = nl;
    v.nf = nf;
    v.n_loc = n_loc;
    v.own0 = own0;
    v.n_own = n_own;
    v.cgeo = cgeo.p;
    v.neigh = neigh.p;
    v.btype = has_btype ? btype.p : nullptr;
    v.tensor = tensor;
    v.blk_start = blk_start.p;
    v.cgid = d_cgid.p;
    v.cell_v0 = sx > 0 ? cell_v0.p : nullptr;
    v.tgeo = sx > 0 ? tgeo.p : nullptr;
    v.tnx = sx;
    v.tny = sy;
    return v;
  }
  void set_device() const { HDD_CUDA(cudaSetDevice(device)); }
  // fills the halo part of a local vector (nd DoFs per cell) from the owning ranks (no-op for world == 1)
  void halo_exchange(double* v_local, int nd);
  ~hdd_mesh();
};

namespace hdd {

struct FnRef {       // index into the device function table, -1 = absent
  int idx = -1;
  int order = 0;
  int kind = 0;      // HDD_FN_*
  bool separable = false;  // expression of the form g(x[0]) * h(x[1])
  bool zero = false; // constant 0: contributes nothing, kernels are skipped
};

struct AffineFn {
  std::vector<FnRef> comps;
  std::vector<std::string> coef_expr;
  std::vector<Program> coef_prog;
  FnRef affine;
  bool has_affine() const { return affine.idx >= 0; }
  bool parametric() const { return !comps.empty(); }
};

struct MgState;  // multigrid.cu
// the preconditioners of the CG solver; the numeric order indexes hdd_swipdg::cg_graph.  mg, mg2 and mg2_simplex are the
// multigrid preconditioners of multigrid.cu: "cg.mg" (Q1 on cubes, P1 on lattice simplices), "cg.mg2" (Q2 on cubes),
// "cg.mg2.simplex" (P2 on lattice simplices)
enum class SolverType { identity, diagonal, blockdiagonal, mg, mg2, mg2_simplex };
constexpr int kNumSolverTypes = int(SolverType::mg2_simplex) + 1;
// block Jacobi and the multigrid types (whose DG-level smoother it is) use the inverses of the cell blocks
inline bool uses_block_inverses(SolverType t) { return t >= SolverType::blockdiagonal; }
inline bool is_multigrid(SolverType t) { return t >= SolverType::mg; }

struct RhsTerm {  // one local functional added into a rhs vector
  int kind;       // 0 L2Volume(f), 1 DirichletBoundarySWIPDG(factor f, g), 2 L2Face(f) on the Neumann faces
  FnRef f, g;
};

struct VectorPart {
  std::string coef_expr;  // empty for the affine part
  Program coef_prog{};
  std::vector<RhsTerm> terms;
  DevBuf<double> values;
};

struct MatrixPart {
  std::string coef_expr;
  Program coef_prog{};
  FnRef factor;
  DevBuf<double> values;
};

// One entry of products_ (discretizations/base.hh:272-291): an affinely decomposed matrix over the system pattern
// ("penalty", "energy") or over the volume pattern ("l2", "h1_semi", "elliptic", "boundary_l2").
struct Product {
  std::string id;
  int which = 0;           // 0 l2, 1 h1_semi, 2 elliptic, 3 boundary_l2, 4 penalty, 5 energy
  bool volume_pattern = true;
  bool assembled = false;
  std::vector<MatrixPart> comps;
  std::unique_ptr<MatrixPart> affine;
};

}  // namespace hdd

struct hdd_swipdg {
  hdd_mesh* mesh = nullptr;
  int polorder = 1;
  int nl = 0;  // local DoFs per cell of the DG space: P1 3, Q1 4, P2 6, Q2 9
  std::vector<int64_t> sub_dof_offsets;  // [n_subdomains+1], mapToGlobal(ss, 0)
  std::string parameter_name;
  int parameter_size = 0;

  hdd::AffineFn factor, force, dirichlet, neumann;
  std::vector<hdd::DevFn> fn_host;
  std::vector<std::unique_ptr<hdd::DevBuf<double>>> fn_cell_storage;
  hdd::DevBuf<hdd::DevFn> fn_dev;
  hdd::DevBuf<double> tensor;
  bool has_tensor = false;

  bool initialized = false;
  std::vector<hdd::MatrixPart> lhs_comps;
  std::unique_ptr<hdd::MatrixPart> lhs_affine;
  std::vector<hdd::VectorPart> rhs_comps;
  std::unique_ptr<hdd::VectorPart> rhs_affine;
  std::vector<const char*> coef_cstr_cache;

  int64_t nnz = 0, n_rows = 0;
  hdd::DevBuf<int64_t> rowptr;
  hdd::DevBuf<int32_t> col;
  // products (only_these_products, discretizations/swipdg.hh:159-163)
  std::vector<std::unique_ptr<hdd::Product>> products;
  std::vector<const char*> product_ids;
  hdd::DevBuf<int64_t> vol_rowptr;
  hdd::DevBuf<int32_t> vol_col;
  hdd::DevBuf<double> prod_frozen, prod_tmp;
  hdd::DevBuf<double> rhs_scratch;  // tables of the tensor-grid rhs path

  // solve workspace
  hdd::DevBuf<double> frozen, dinv, dinv_block, z, b, x, r, p, q, partial, tmp_local;
  // peer-memory SpMV (multi GPU): ping-pong direction, dinv with halo, peers' r / p buffers mapped through CUDA IPC
  hdd::DevBuf<double> p_alt, dinv_local;
  bool p2p_ready = false, p2p_failed = false;
  hdd::PeerView peer_view{};
  std::vector<void*> ipc_opened;
  hdd::SolverType last_type = hdd::SolverType::diagonal;  // of the last hdd_solve
  hdd::MgState* mg = nullptr;
  // CUDA graph of two CG iterations, cached per solver type; valid while the operator / workspace pointers it was
  // captured with are the ones in use (cg_graph_key)
  struct CgGraph {
    cudaGraphExec_t exec = nullptr;
    const void* key[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    int64_t launches = 0;
  };
  CgGraph cg_graph[hdd::kNumSolverTypes];
  hdd::DevBuf<hdd::CgScalars> sc;
  hdd::CgScalars* sc_host = nullptr;  // pinned
  bool have_solution = false;

  // estimator workspace
  hdd::DevBuf<double> vertex_mean, ind_out, seg_out;
  bool estimator_vector_resident = false;        // tmp_local holds the vector of the last hdd_estimate (halo included)
  const hdd_parameters* profile_prm = nullptr;   // parameters hdd_profile_kernel(4/5) evaluates the estimator at

  hdd::MeshView view() const {
    hdd::MeshView v = mesh->view(has_tensor ? tensor.p : nullptr);
    v.nl = nl;
    return v;
  }
  const hdd::DevFn* fn(const hdd::FnRef& r) const { return fn_dev.p + r.idx; }
  const hdd::DevFn& fn_h(const hdd::FnRef& r) const { return fn_host[size_t(r.idx)]; }
  ~hdd_swipdg();
};

namespace hdd {
// shared by swipdg.cu and products.cu
void require_init(const hdd_swipdg* h);                                          // assert_everything_is_ready (base.hh:370-377)
void check_mu(const hdd_swipdg* h, const double* mu, int mu_size, const char* name);  // base.hh:333-334
double eval_coef(const Program& p, const double* mu, int mu_size);
void assemble_products(hdd_swipdg* h);
// multigrid.cu ("cg.mg", "cg.mg2", "cg.mg2.simplex")
void mg_detect_structure(hdd_mesh* m, const double* xy_host, const double* xy_dev, int64_t v_begin, int64_t v_end,
                         const int32_t* cv_dev, int64_t n_verts);
void mg_setup(hdd_swipdg* h, const double* frozen_values, SolverType type);
void mg_apply(hdd_swipdg* h, const int* done, const double* r, double* z, double* p_init, double* partial, CgScalars* sc);
void mg_release(MgState* st);
// copies the finest level's V-cycle results of the last mg_apply, n_hier (nx+1)(ny+1) doubles, on the handle's stream
void mg_vertex_result(const hdd_swipdg* h, double* host);
int mg_num_levels(const hdd_swipdg* h);  // the product assemblers added to system_assembler (discretizations/swipdg.hh:359-479)
DevCombo make_combo(const hdd_swipdg* h, const AffineFn& f, const double* mu, int mu_size);  // f frozen at mu
}  // namespace hdd
