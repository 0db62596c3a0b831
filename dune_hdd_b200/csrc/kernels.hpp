// Host-callable launchers of the sm_100a kernels (K1..K10 of SURVEY.md 8a).
#pragma once
#include <cuda_runtime.h>

#include "device.cuh"

namespace hdd {

// ---- K0: device-side localisation of the host grid -------------------------------------------------------------------
// cgeo[c] from (xy, cell_verts); xy is addressed by global vertex id and valid in [v_begin, v_end); flag |= 1 if a cube
// cell is not an axis-parallel rectangle (also validates the vertex ids: flag |= 4 if one is outside that range)
void launch_build_geometry(int kind, int32_t n_loc, int32_t v_begin, int32_t v_end, const double* xy, const int32_t* cell_verts_local,
                           double* cgeo, int32_t* flag, cudaStream_t s);
// A structured nx x ny grid on [x0,x1] x [y0,y1] with px x py boxes as subdomains, cells numbered subdomain-major (boxes x
// fastest, cells inside a box x fastest): X[px+1] / Y[py+1] first cell column / row of every box, off[px*py+1] first cell id
// of every box (device arrays).
struct CubeGridDesc {
  int nx, ny, px, py;
  double x0, x1, y0, y1;
  const int32_t* X;
  const int32_t* Y;
  const int64_t* off;
};
// fills cgeo / cell_v0 / lex_cell / cgid for the local cells [lower halo | owned | upper halo] and the global face-neighbour
// ids of the owned cells, plus the one-dimensional geometry tables
void launch_cube_fill(const CubeGridDesc& g, int32_t n_loc, int32_t own0, int32_t n_own, int32_t cell_begin, const int32_t* halo,
                      double* cgeo, int32_t* cell_v0, int32_t* lex_cell, int32_t* cgid, int32_t* neigh, double* tgeo,
                      cudaStream_t s);
// whole mesh on one GPU: flag |= 8 if a neighbour id is out of range; out[i] = i
void launch_validate_neighbours(const int32_t* neigh, int64_t count, int32_t n_cells, int32_t* flag, cudaStream_t s);
void launch_iota(int32_t* out, int32_t n, cudaStream_t s);
void launch_iota_from(int32_t* out, int32_t n, int32_t first, cudaStream_t s);  // out[i] = first + i
// subdomain offsets and neighbouring-subdomain byte matrix of a whole mesh; flag |= 16 if not subdomain-major
void launch_subdomain_structure(const int32_t* sub, const int32_t* neigh, int nf, int32_t n_cells, int n_sub,
                                int64_t* offsets, uint8_t* adj, int32_t* flag, cudaStream_t s);
// in place: global neighbour ids of the owned cells -> local ids ([lower halo | owned | upper halo]); flag |= 2 if missing
void launch_localize_neighbours(int32_t* neigh, int64_t count, int32_t cell_begin, int32_t cell_end, const int32_t* halo,
                                int32_t n_lo, int32_t n_hi, int32_t* flag, cudaStream_t s);

// ---- K1: pattern ------------------------------------------------------------------------------------------
// nblk[k] = number of blocks of owned cell k (1 + #neighbours); blk_start is its exclusive prefix sum.
void launch_count_blocks(const MeshView& m, int64_t* nblk, cudaStream_t s);
void exclusive_scan_i64(const int64_t* in, int64_t* out, int64_t n, cudaStream_t s);
void launch_fill_csr(const MeshView& m, int64_t* rowptr, int32_t* col, cudaStream_t s);

// ---- K2/K3: assembly ----------------------------------------------------------------------------------------
// one affine part of the system matrix: values in CSR order of the owned rows.  Function descriptors travel by value
// (kernel parameter space = constant bank), so the expression programs are never fetched from global memory.
void launch_assemble_lhs(const MeshView& m, const DevFn& factor_dev, int factor_kind, int factor_order, int polorder,
                         double* values, cudaStream_t s);
// the penalty terms only (Products::SwipdgPenaltyAssemblable, over_integrate = 2), same pattern as the system matrix
void launch_assemble_penalty(const MeshView& m, const DevFn& factor_dev, int factor_kind, int factor_order, int polorder,
                             double* values, cudaStream_t s);
// volume-pattern products, values [n_own * nl * nl] (one dense block per cell): which = 0 l2, 1 h1_semi, 2 elliptic,
// 3 boundary_l2 (discretizations/swipdg.hh:359-443)
void launch_assemble_block_product(const MeshView& m, int which, const DevFn& factor_dev, int factor_order, int polorder,
                                   double* values, cudaStream_t s);
// A logically structured (tensor-product) cube grid as the mesh detected it: cells per direction, vertex 0 of every
// local cell, and scratch for the per-column / per-row tables of the separable-force fast path
// (>= (nx + ny) * (2 + p + 1) doubles).
struct TensorGridView {
  int nx = 0, ny = 0;
  const int32_t* cell_v0 = nullptr;
  double* scratch = nullptr;
};
// b (+)= L2Volume(force).  accumulate = false overwrites b (no memset, no read-modify-write for the first term)
void launch_rhs_volume(const MeshView& m, const DevFn& force_dev, int force_order, bool separable, int polorder,
                       bool accumulate, const TensorGridView* tg, double* b, cudaStream_t s);
// b += DirichletBoundarySWIPDG(factor, tensor, dirichlet)
void launch_rhs_dirichlet(const MeshView& m, const DevFn& factor_dev, int factor_order, const DevFn& dirichlet_dev,
                          int dirichlet_order, int polorder, double* b, cudaStream_t s);

// b += L2Face(neumann) on the Neumann faces
void launch_rhs_neumann(const MeshView& m, const DevFn& neumann_dev, int neumann_order, int polorder, double* b,
                        cudaStream_t s);

// ---- K4: freeze -----------------------------------------------------------------------------------------------
// out = sum_k theta[k] * parts[k]   (values-only AXPY over a shared pattern, discretizations/base.hh:349-361)
struct FreezeArgs {
  int n;
  double theta[kMaxParts];
  const double* part[kMaxParts];
};
void launch_freeze(const FreezeArgs& a, double* out, int64_t count, cudaStream_t s);
// dinv[row] = 1 / A[row,row] (Jacobi) or 1 (identity)
void launch_extract_dinv(const MeshView& m, const double* values, int jacobi, double* dinv, cudaStream_t s);
void launch_invert_diag_blocks(const MeshView& m, const double* values, double* dinv_block, cudaStream_t s);

// ---- K5/K6: CG ---------------------------------------------------------------------------------------------------
struct CgScalars {     // device resident, ping-pong indexed by iteration parity
  double rz[2];
  int done[2];
  int it[2];
  double pq;           // p.Ap of the current iteration (after reduction / all-reduce)
  double rz_new;       // r.z after the update
  double rr;           // r.r after the update
  double bb;           // b.b
  double tol2;         // precision^2
  int max_it;
  unsigned int ticket_a, ticket_b;  // last-block tickets
  double red[4];       // all-reduce staging: [0] pq, [1] rz_new, [2] rr
};

struct CgBuffers {
  const double* values;  // frozen operator, CSR order
  const double* dinv;    // owned rows (identity / diagonal preconditioner)
  const double* dinv_block;  // [n_own * nl * nl] inverted diagonal blocks (block Jacobi) or nullptr
  double* z;             // owned rows, preconditioned residual (block Jacobi only) or nullptr
  const double* b;       // owned rows
  double* x;             // owned rows
  double* r;             // owned rows
  double* p;             // LOCAL vector (halo | owned | halo); parity-0 buffer when p_alt != nullptr
  double* p_alt;         // parity-1 direction buffer (ping-pong, peer-memory mode) or nullptr
  double* q;             // owned rows
  double* partial;       // >= 3 * max_blocks
  CgScalars* sc;
};

// Peer-memory view for the fused SpMV + halo read (multi GPU, Q1): the halo part of the CG direction is never
// exchanged; the kernel reads the owner's r and previous direction through NVLink and forms p = D^-1 r + beta p_old on
// the fly.  The two all-reduces of the CG iteration are the only synchronisation (see DESIGN.md 7).
constexpr int kMaxPeers = 16;
struct PeerView {
  int enabled;
  int own0, n_own;               // of this rank
  const int32_t* halo_peer;      // [n_halo] owner rank
  const int32_t* halo_rcell;     // [n_halo] cell offset inside the owner's owned range
  const double* dinv_local;      // [n_loc * nl] Jacobi diagonal inverse including the halo
  const double* r[kMaxPeers];    // owners' residuals (owned rows)
  const double* p[2][kMaxPeers]; // owners' direction buffers (local vectors) by parity
  int own0_of[kMaxPeers];        // owners' own0
};

int cg_partial_capacity();
bool cg_spmv_uses_tma(const MeshView& m);  // the peer-memory halo read lives in the TMA SpMV kernel
// y = A x over the owned rows; x is a local vector.  If partial != nullptr also writes per-block partial sums of
// x_owned . y and, through the last-block ticket, their total into sc->pq / sc->red[0].
void launch_spmv(const MeshView& m, const double* values, const double* x_local, double* y, cudaStream_t s);
void launch_cg_init(const MeshView& m, const CgBuffers& c, double precision, int max_it, cudaStream_t s);
void launch_cg_init_finish(const MeshView& m, const CgBuffers& c, cudaStream_t s);
void launch_cg_spmv(const MeshView& m, const CgBuffers& c, int parity, cudaStream_t s, const PeerView* peer = nullptr);
void launch_cg_update(const MeshView& m, const CgBuffers& c, int parity, cudaStream_t s);
void launch_cg_direction(const MeshView& m, const CgBuffers& c, int parity, cudaStream_t s);

// sc->red[0] = sum (b - q)^2, red[1] = sum b^2, red[2] = sum x^2 over n entries, red[3] = max |values| (hdd_residual)
void launch_residual_norms(const double* b, const double* q, const double* x, int64_t n, const double* values, int64_t nnz,
                           double* partial, CgScalars* sc, cudaStream_t s);

// a15 (pure Neumann): symmetric unit row/column 0 + rhs[0] = 0, and x -= mean(x) after the solve
void launch_unit_row_col0(const MeshView& m, double* values, double* b, cudaStream_t s);
void launch_subtract_mean(double* x, int64_t n, double* partial, CgScalars* sc, cudaStream_t s);

// ---- K7-K10: estimators ---------------------------------------------------------------------------------------
struct IndicatorArgs {
  DevCombo a_mu, a_hat, a_bar, a_cut, a_min, a_max;
  const DevFn* fn_table;       // the handle's function table (global memory); staged in shared memory by the kernel
  int n_fn;
  int force_idx;
  int force_order;
  const double* u_local;       // local vector
  const double* vertex_mean;   // [n_verts_local], Oswald values (0 on the boundary)
  const int32_t* cell_verts;   // [n_own*3] local vertex ids
  double* out;                 // [9][n_own]: nc2,res2,r2,df2,dfstar2,rstar2,amin,resstar2,esv2
};
void launch_oswald_vertex_means(const int64_t* vptr, const int32_t* vdof, const uint8_t* vboundary, int32_t n_verts,
                                const double* u_local, double* vertex_mean, cudaStream_t s);
// fn_table_host: the host copy of a.fn_table (decides whether any diffusion-factor part is an expression)
void launch_indicators(const MeshView& m, const IndicatorArgs& a, const DevFn* fn_table_host, int polorder, cudaStream_t s);
// deterministic segmented reductions (fixed trees): out[r * n_seg + seg] = sum (or min, if bit r of min_mask is set)
// over k in [seg_ptr[seg], seg_ptr[seg+1]) of in[r * row_stride + k], all rows in one launch
void launch_segment_reduce(const double* in, int64_t row_stride, int n_rows, unsigned min_mask, const int64_t* seg_ptr_dev,
                           int n_seg, double* out, cudaStream_t s);
void launch_segment_sums(const double* in, const int64_t* seg_ptr_dev, int n_seg, double* out, cudaStream_t s);
void launch_segment_min(const double* in, const int64_t* seg_ptr_dev, int n_seg, double* out, cudaStream_t s);

// ---- K12/K13: products in use, error norms ---------------------------------------------------------------------
void launch_fill_volume_csr(const MeshView& m, int64_t* rowptr, int32_t* col, cudaStream_t s);
// y = P x for a volume-pattern (block diagonal) product; x and y over the owned rows
void launch_block_spmv(const MeshView& m, const double* values, const double* x_own, double* y, cudaStream_t s);
// out[3][n_own]: per cell int (u_h-u)^2, int |grad(u_h-u)|^2, int a K grad(u_h-u).grad(u_h-u) with a rule of `order`
void launch_error_norms(const MeshView& m, int polorder, const DevFn& exact, const DevFn& exact_dx, const DevFn& exact_dy,
                        const DevCombo& factor, const DevFn* fn_table, int order, const double* u_own, double* out,
                        cudaStream_t s);
// out[seg] = sum over the DoFs of the cells [seg_ptr[seg], seg_ptr[seg+1]) of x * y
// Operators::Prolongation: u_fine (owned cells of `fine`) = the coarse DG function at the fine Lagrange nodes; father =
// coarse cell id per owned fine cell, cgeo_coarse = geometry records of a whole (non-distributed) coarse mesh; *flag is
// set if a father id is out of range
void launch_prolong(const MeshView& fine, int p_fine, const double* cgeo_coarse, int32_t n_coarse, int p_coarse,
                    const int32_t* father, const double* u_coarse, double* u_fine, int* flag, cudaStream_t s);
void launch_segment_dot(const double* x, const double* y, const int64_t* seg_ptr_dev, int n_seg, int nd, double* out,
                        cudaStream_t s);

// ---- K11: halo pack --------------------------------------------------------------------------------------------
// out[k * nd + i] = v_local[cells[k] * nd + i]: the DoFs of the listed local cells, nd DoFs per cell
void launch_pack(const double* v_local, const int32_t* cells, int64_t n_cells, int nd, double* out, cudaStream_t s);

}  // namespace hdd
