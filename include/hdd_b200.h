/*
 * hdd_b200.h - C-ABI of the B200-native SWIPDG hot path (assembly -> CG solve -> estimators).
 *
 * This is the drop-in boundary for dune-hdd's LinearElliptic::Discretizations::SWIPDG /
 * BlockSWIPDG and LinearElliptic::Estimators::{SWIPDG,BlockSWIPDG}.  The reference has no
 * FFI of its own (its seam is a C++ template API plus a pybindgen projection), so every entry
 * point below cites the reference method it replaces; INTEGRATION.md shows the C++ facade and
 * the Python binding a dune-hdd maintainer would put on top.
 *
 * Conventions
 *  - plain pointers and sizes only; every function returns an hdd_status (0 = ok) and leaves a
 *    message retrievable through hdd_last_error() (thread local).
 *  - all numbers are fp64 (RangeFieldType = double, testcases/ESV2007.hh:37); cell / DoF indices are
 *    int32 (cells) and int64 (matrix offsets).
 *  - "host" pointers are ordinary host memory, "dev" pointers are CUDA device memory owned by
 *    the handle they were obtained from and valid until that handle is destroyed.
 *  - one host thread per handle; all work of a handle is ordered on the handle's CUDA stream
 *    (the reference objects are not thread safe either: mutable cache_, discretizations/base.hh:192).
 *  - there is no CPU fallback: without a CUDA device hdd_mesh_create fails with HDD_ERR_DEVICE.
 *
 * Citations `file:line` are relative to the dune-hdd tree; `dune/hdd/linearelliptic/` is omitted.
 */
#ifndef HDD_B200_H
#define HDD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes: one per exception type the reference throws on this path --------------- */
typedef enum hdd_status {
  HDD_OK = 0,
  HDD_ERR_WRONG_INPUT = 1,          /* Stuff::Exceptions::wrong_input_given        (discretizations/base.hh:289) */
  HDD_ERR_USING_THIS_WRONG = 2,     /* Stuff::Exceptions::you_are_using_this_wrong (discretizations/base.hh:373, estimators/swipdg.hh:968) */
  HDD_ERR_WRONG_PARAMETER_TYPE = 3, /* Pymor::Exceptions::wrong_parameter_type     (discretizations/base.hh:333-334) */
  HDD_ERR_INDEX_OUT_OF_RANGE = 4,   /* Stuff::Exceptions::index_out_of_range       (discretizations/block-swipdg.hh:560-562) */
  HDD_ERR_NOT_IMPLEMENTED = 5,      /* Dune::NotImplemented                        (discretizations/swipdg.hh:173-176) */
  HDD_ERR_REQUIREMENTS_NOT_MET = 6, /* Stuff::Exceptions::requirements_not_met     (estimators/block-swipdg.hh:766-773) */
  HDD_ERR_INTERNAL = 7,             /* Stuff::Exceptions::internal_error */
  HDD_ERR_DEVICE = 8,               /* CUDA / NCCL failure, or no device */
  HDD_ERR_NOT_CONVERGED = 9         /* Stuff::Exceptions::linear_solver_failed (upstream Stuff::LA::Solver) */
} hdd_status;

const char* hdd_last_error(void);
const char* hdd_version(void);

/* ---- grids ------------------------------------------------------------------------------- */
/* Element kinds.  Vertex and face numbering follow the Dune reference elements
 *   HDD_SIMPLEX2D: vertices (0,0),(1,0),(0,1);       faces {0,1},{0,2},{1,2}
 *   HDD_CUBE2D   : vertices (0,0),(1,0),(0,1),(1,1); faces {0,2},{1,3},{0,1},{2,3}  (axis-parallel cells only)
 * The DG space is GDT::Spaces::DiscontinuousLagrangeProvider (discretizations/swipdg.hh:94-95):
 * global DoF = n_loc * cell + local vertex index, n_loc = 3 (P1) resp. 4 (Q1). */
enum { HDD_SIMPLEX2D = 0, HDD_CUBE2D = 1 };

typedef struct hdd_mesh hdd_mesh;

/* Replaces the grid view + boundary info + (for BlockSWIPDG) the ms_grid handed to
 * SWIPDG(grid_provider, boundary_info_cfg, problem, level) (discretizations/swipdg.hh:159-163) and
 * BlockSWIPDG(ms_grid_provider, ...) (discretizations/block-swipdg.hh:172-176).
 *   xy             [2*n_verts]        vertex coordinates
 *   cell_verts     [n_loc*n_cells]    vertex ids, reference-element order
 *   cell_neigh     [n_faces*n_cells]  neighbour cell across each face, -1 = domain boundary
 *   cell_subdomain [n_cells] or NULL  subdomain of each cell (grid::Multiscale::subdomainOf); cells must be
 *                                     numbered subdomain-major so that the global DoF index equals
 *                                     Spaces::Block::mapper().mapToGlobal(ss, i) (discretizations/block-swipdg.hh:1042)
 *   boundary_type  [n_faces*n_cells] or NULL   1 = Dirichlet (default, AllDirichlet), 2 = Neumann
 * The arrays are copied; the caller may free them afterwards.  Vertex and neighbour ids are validated (on the device
 * for a whole mesh): HDD_ERR_INDEX_OUT_OF_RANGE.  A HDD_CUBE2D grid whose vertices are numbered x-fastest over a
 * tensor-product coordinate grid (Stuff::Grid::Providers::Cube< SGrid >, hdd_grid_cube) is recognised as logically
 * structured; assembly then reads its cell sizes from per-column / per-row tables and the solver type "cg.mg" is
 * available.
 * rank / world_size: this process owns the contiguous cell range [cell_begin, cell_end) (whole subdomains);
 * pass 0, 1, 0, n_cells for a single GPU.  device = CUDA ordinal. */
int hdd_mesh_create(int kind, int64_t n_cells, int64_t n_verts, const double* xy, const int32_t* cell_verts,
                    const int32_t* cell_neigh, const int32_t* cell_subdomain, const uint8_t* boundary_type,
                    int64_t cell_begin, int64_t cell_end, int device, hdd_mesh** out);
/* Stuff::Grid::Providers::Cube< SGrid<2,2> >(lower_left, upper_right, num_elements) with the [px py 1] partition of
 * grid::Multiscale, the way the reference's structured test cases get their grids (testcases/ESV2007.hh:123-127, :150-163;
 * testcases/spe10.hh:262-268, :301-307): nothing but these numbers travels to the device, where one kernel writes the
 * geometry, neighbour and numbering tables of the cells this rank keeps.  Same grid, same subdomain-major cell numbering,
 * bit-identical coordinates as hdd_grid_cube + hdd_mesh_create (tests compare the assembled matrices).  cell_end < 0 means
 * "all cells"; the owned range must consist of whole subdomains. */
int hdd_mesh_create_cube(int64_t nx, int64_t ny, double x0, double x1, double y0, double y1, int px, int py,
                         int64_t cell_begin, int64_t cell_end, int device, hdd_mesh** out);
int hdd_mesh_destroy(hdd_mesh* mesh);
/* Page-locked host memory for the grid / solution arrays handed to this library: copies from and to it run at PCIe /
 * NVLink-C2C speed instead of being staged through the driver's bounce buffers (4096^2 grid: 0.87 GB of arrays).
 * Ordinary host memory works everywhere, it is only slower.  Release with hdd_host_free. */
int hdd_host_alloc(size_t bytes, void** ptr);
int hdd_host_free(void* ptr);
int hdd_mesh_num_cells(const hdd_mesh* mesh, int64_t* n_global, int64_t* n_owned, int64_t* n_halo);

/* Stand-ins for Stuff::Grid::Providers::Cube<GridType>(lower_left, upper_right, num_elements) as used by the
 * test cases (testcases/ESV2007.hh:123-127, testcases/spe10.hh:262-268): host-side generators that fill caller
 * arrays.  hdd_grid_cube: nx*ny axis-parallel cells, x fastest (SGrid).  hdd_grid_simplex: the conforming
 * ALUGrid<2,2,simplex,conforming> ladder obtained from n x n squares after an even number of uniform bisections:
 * squares_per_side^2 squares, each cut into 8 right triangles around its centre (8*s^2 cells).
 * partitions_x/y > 1 renumber the cells subdomain-major ([px py 1] partition, testcases/ESV2007.hh:150-163) and
 * fill cell_subdomain (may be NULL otherwise). */
int hdd_grid_cube_sizes(int64_t nx, int64_t ny, int64_t* n_cells, int64_t* n_verts);
int hdd_grid_cube(int64_t nx, int64_t ny, double x0, double x1, double y0, double y1, int partitions_x,
                  int partitions_y, double* xy, int32_t* cell_verts, int32_t* cell_neigh, int32_t* cell_subdomain);
int hdd_grid_simplex_sizes(int64_t squares_per_side, int64_t* n_cells, int64_t* n_verts);
int hdd_grid_simplex(int64_t squares_per_side, double x0, double x1, double y0, double y1, int partitions_x,
                     int partitions_y, double* xy, int32_t* cell_verts, int32_t* cell_neigh,
                     int32_t* cell_subdomain);
/* Father cell of every cell of a finer grid covering the same domain: the coarse cell that contains the fine cell's
 * centre.  The reference walks ALUGrid's father() links (test/linearelliptic-swipdg.hh:186-194) or searches the coarse
 * grid view with Stuff::Grid::EntityInlevelSearch (test/linearelliptic-block-swipdg.hh:169-177); on flat arrays it is a
 * bucketed point location (host, threaded, no device).  father: n_fine entries.  HDD_ERR_WRONG_INPUT if a centre lies
 * in no coarse cell. */
int hdd_grid_fathers(int kind, int64_t n_coarse, int64_t n_coarse_verts, const double* xy_coarse,
                     const int32_t* cell_verts_coarse, int64_t n_fine, int64_t n_fine_verts, const double* xy_fine,
                     const int32_t* cell_verts_fine, int32_t* father);

/* ---- problem data (ProblemInterface, problems/interfaces.hh:84-144) ----------------------------------- */
/* A scalar data function as the host sees it after localisation:
 *   HDD_FN_CONSTANT   Stuff::Functions::Constant                         -> value
 *   HDD_FN_CELLWISE   piecewise constant (Spe10::Model1, Indicator, Checkerboard evaluated per cell by the
 *                     host from the DUNE function object)                -> cell_values[n_cells] (global numbering)
 *   HDD_FN_EXPRESSION Stuff::Functions::Expression("x", expr, order)     -> expression in x[0], x[1], pi
 *                     (problems/OS2014.hh:63-74); ESV2007::Testcase1Force is "0.5*pi*pi*cos(0.5*pi*x[0])*cos(0.5*pi*x[1])"
 * `order` is the polynomial order the function reports (drives the quadrature rule exactly as in dune-gdt). */
enum { HDD_FN_CONSTANT = 0, HDD_FN_CELLWISE = 1, HDD_FN_EXPRESSION = 2 };

typedef struct hdd_function {
  int kind;
  int order;
  double value;
  const double* cell_values;
  const char* expression;
} hdd_function;

/* Pymor::Functions::AffinelyDecomposableDefault: sum_q theta_q(mu) * component_q + affine_part.
 * coefficients[q] is the Pymor::ParameterFunctional expression in `mu` (e.g. "mu", "-1.0*mu"). */
typedef struct hdd_affine_function {
  int n_components;
  const hdd_function* components;
  const char* const* coefficients;
  const hdd_function* affine_part; /* NULL = none */
} hdd_affine_function;

typedef struct hdd_problem {
  hdd_affine_function diffusion_factor;
  const double* diffusion_tensor; /* [4*n_cells] row-major 2x2 per cell (global numbering), NULL = identity;
                                     never parametric (discretizations/swipdg.hh:173-176) */
  hdd_affine_function force;
  hdd_affine_function dirichlet;
  hdd_affine_function neumann;
  const char* parameter_name; /* "mu" (problems/OS2014.hh:72), NULL if non-parametric */
  int parameter_size;         /* 1 */
} hdd_problem;

/* ---- discretization ---------------------------------------------------------------------------- */
typedef struct hdd_swipdg hdd_swipdg;

enum { HDD_LHS = 0, HDD_RHS = 1 };

/* SWIPDG::SWIPDG(...) (discretizations/swipdg.hh:159-177) / BlockSWIPDG::BlockSWIPDG (block-swipdg.hh:172-260).
 * polorder = 1 (P1 / Q1, n_loc = 3 / 4) or 2 (P2 / Q2, n_loc = 6 / 9; nodes in lexicographic order - (0,0),(1/2,0),(1,0),
 * (0,1/2),(1/2,1/2),(0,1) on the triangle, i + 3 j on the square; unpinned: every reference test instantiates polOrder 1,
 * test/linearelliptic-swipdg.cc:45).  The estimators need polorder 1.  Fails with HDD_ERR_WRONG_INPUT if the factor is
 * empty etc. */
int hdd_swipdg_create(hdd_mesh* mesh, int polorder, const hdd_problem* problem, hdd_swipdg** out);
int hdd_swipdg_destroy(hdd_swipdg* h);

/* SWIPDG::init() (discretizations/swipdg.hh:206-512): all affine parts of the system matrix (on the block-compressed
 * pattern, see hdd_pattern) and of the rhs, assembled on the GPU in one pass per part set.  Idempotent
 * (container_based_initialized_, :208,:510). */
int hdd_swipdg_init(hdd_swipdg* h);
/* Re-runs only system_assembler.walk() (:485) on an initialised handle; used by the benchmark. seconds may be NULL. */
int hdd_swipdg_assemble(hdd_swipdg* h, double* seconds);

int hdd_num_dofs(const hdd_swipdg* h, int64_t* n_global, int64_t* n_owned);   /* space.mapper().size() */
/* pattern() (discretizations/swipdg.hh:201-204) as CSR of the owned rows; col holds global DoF indices.  The library keeps
 * the pattern in block-compressed form (block offsets per cell + the neighbour table, built with the mesh); the expanded
 * index arrays are written on the device at the first call that asks for rowptr_dev or col_dev and kept from then on. */
int hdd_pattern(hdd_swipdg* h, int64_t* n_rows, int64_t* nnz, const int64_t** rowptr_dev, const int32_t** col_dev);
/* system_matrix()/rhs() parts (discretizations/base.hh:240-270): num_components(), component(q), coefficient(q),
 * has_affine_part(), affine_part().  q = -1 addresses the affine part. */
int hdd_num_components(const hdd_swipdg* h, int which, int* n_components, int* has_affine_part);
int hdd_component_values(hdd_swipdg* h, int which, int q, const double** values_dev, int64_t* count);
int hdd_component_coefficient(const hdd_swipdg* h, int which, int q, const char** expression);
/* evaluates the coefficients theta_q(mu) of `which` (ParameterFunctional::evaluate). */
int hdd_evaluate_coefficients(const hdd_swipdg* h, int which, const double* mu, int mu_size, double* theta);
int hdd_copy_to_host(hdd_swipdg* h, void* dst_host, const void* src_dev, size_t bytes);
int hdd_sync(hdd_swipdg* h);

/* get_operator().freeze_parameter(mu).apply(x, y) - one SpMV with the frozen operator (block-swipdg.hh:741). */
int hdd_apply(hdd_swipdg* h, const double* mu, int mu_size, const double* x_host, double* y_host);
/* True relative residual ||b(mu) - A(mu) x||_2 / ||b(mu)||_2 of the solution the last hdd_solve left on the device,
 * recomputed from scratch (one SpMV with the frozen operator, global over all ranks): what a caller of the reference would
 * get from rhs - system_matrix.mv(solution) after solve() (discretizations/base.hh:361-364).  Collective on N GPUs.
 * fp64_floor (nullable): the size of that quantity's own rounding error, 2^-53 (1 + n_faces) n_loc max|A_ij| ||x|| / ||b||
 * - the right-hand side of the SWIPDG system scales with h^2 against O(1) matrix entries, so on fine grids a recomputed
 * residual cannot fall below it however long the solver iterates (4096^2 Q1: a few 1e-9). */
int hdd_residual(hdd_swipdg* h, const double* mu, int mu_size, double* relative_residual, double* fp64_floor);

typedef struct hdd_solve_info {
  int iterations;
  int converged;
  double relative_residual; /* ||r||_2 / ||b||_2 (recursive) */
  double seconds;           /* device time of freeze + CG, CUDA events */
  double seconds_per_iteration;
  int peer_memory;          /* multi GPU: 1 = fused SpMV + halo read over peer memory (NVLink), 0 = NCCL send/recv */
} hdd_solve_info;

/* solver_types() / solver_options(type) (discretizations/base.hh:314-322). Types: "cg.diagonal" (default,
 * Jacobi), "cg.blockdiagonal" (block Jacobi with the n_loc x n_loc cell blocks), "cg.identity", and "cg.mg": CG with
 * a two-level preconditioner (block Jacobi + conforming-Q1 / P1 coarse space solved by geometric multigrid V-cycles,
 * the counterpart of the AMG-preconditioned default of the reference's Stuff::LA::Solver) - polOrder 1 on logically
 * structured grids: HDD_CUBE2D with the vertices numbered x-fastest, or a simplex grid whose vertices form such a
 * lattice and whose triangles join lattice neighbours; and "cg.mg2": the same for polOrder 2 (block Jacobi with the
 * 9 x 9 cell blocks + conforming Q1 + the Q2 hourglass family, one V-cycle each) - Q2 on logically structured
 * HDD_CUBE2D grids only.  Elsewhere both give HDD_ERR_REQUIREMENTS_NOT_MET.  Aliases "cg", "cg.jacobi",
 * "cg.diagonal.lower", "cg.identity.lower", "cg.blockjacobi", "cg.multigrid", "cg.multigrid2". */
int hdd_solver_types(const char* const** types, int* n_types);
/* uncached_solve(options, vector, mu) (discretizations/base.hh:327-367): freeze lhs and rhs at mu, CG.
 * precision / max_iter mirror Stuff::LA::Solver's option keys.  x_host[n_owned] receives the solution
 * (NULL: keep it on the device only, see hdd_solution_dev).  mu may be NULL for non-parametric problems;
 * a wrong mu_size gives HDD_ERR_WRONG_PARAMETER_TYPE (:333-334). */
int hdd_solve(hdd_swipdg* h, const char* type, double precision, int max_iter, const double* mu, int mu_size,
              double* x_host, hdd_solve_info* info);
int hdd_solution_dev(hdd_swipdg* h, const double** x_dev);

/* ---- products (discretizations/swipdg.hh:359-508, block-swipdg.hh:392-548, base.hh:272-291) ---------------- */
/* The `only_these_products` constructor argument (discretizations/swipdg.hh:159-163): ids out of "l2", "h1_semi",
 * "elliptic", "boundary_l2", "penalty", "energy" (others are ignored, like the std::find tests of :364-505).  Call
 * before hdd_swipdg_init (they are then assembled by init() together with the system, like in system_assembler.walk());
 * on an initialised handle they are assembled at once.  Default: none, as in the reference.
 *   l2           int_T phi_i phi_j                             volume pattern (one dense n_loc x n_loc block per cell)
 *   h1_semi      int_T grad phi_j . grad phi_i                 volume pattern
 *   elliptic     int_T a_q K grad phi_j . grad phi_i           volume pattern, one part per diffusion-factor part
 *   boundary_l2  int_{dT on dOmega} phi_i phi_j                volume pattern
 *   penalty      the penalty terms of the SWIPDG form only     system pattern (hdd_pattern), one part per factor part
 *   energy       copy of the system matrix                     system pattern (aliases hdd_component_values(HDD_LHS))
 * all with over_integrate = 2 (:359). */
int hdd_swipdg_only_these_products(hdd_swipdg* h, const char* const* ids, int n);
/* available_products() (discretizations/base.hh:272-280), sorted like the std::map. */
int hdd_products_available(const hdd_swipdg* h, const char* const** ids, int* n);
/* get_product(id) (base.hh:281-291): HDD_ERR_USING_THIS_WRONG if there are no products, HDD_ERR_WRONG_INPUT for an
 * unknown id.  volume_pattern: 1 = values follow hdd_pattern_volume, 0 = hdd_pattern.  q = -1 is the affine part. */
int hdd_product_num_components(hdd_swipdg* h, const char* id, int* n_components, int* has_affine_part, int* volume_pattern);
int hdd_product_values(hdd_swipdg* h, const char* id, int q, const double** values_dev, int64_t* count);
int hdd_product_coefficient(hdd_swipdg* h, const char* id, int q, const char** expression);
int hdd_pattern_volume(hdd_swipdg* h, int64_t* n_rows, int64_t* nnz, const int64_t** rowptr_dev, const int32_t** col_dev);
/* get_product(id).freeze_parameter(mu).apply2(u, v) = u^T P(mu) v on the device (u, v: owned rows; all ranks call it
 * collectively and receive the global value).  The induced norm is sqrt(apply2(u, u)). */
int hdd_product_apply2(hdd_swipdg* h, const char* id, const double* mu, int mu_size, const double* u_host,
                       const double* v_host, double* result);
/* Error norms of the convergence studies (test/linearelliptic-swipdg.hh:267-290: Products::L2 / H1Semi / Elliptic induced
 * norms of the difference) against an analytic solution given as Expression strings in x[0], x[1] for u, du/dx, du/dy;
 * evaluated on this grid with the element rule exact for `order`; out3 = {L2, H1_semi, energy}, global over all ranks.
 * u_host = NULL uses the last solution. */
int hdd_error_norms(hdd_swipdg* h, const double* u_host, const char* exact, const char* exact_dx, const char* exact_dy,
                    int order, const double* mu, int mu_size, double* out3);
/* GDT::Operators::Prolongation(reference_grid_view).apply(coarse_function, fine_function) of the convergence studies
 * (test/linearelliptic.hh:168-176): every DoF of the fine DG function becomes the value of the coarse DG function at the
 * fine Lagrange node.  father[k] = the coarse cell containing owned fine cell k (hdd_grid_fathers).  The coarse
 * discretization must own its whole grid and live on the same device; the fine one may be distributed (u_fine = its
 * owned rows); the polynomial orders may differ.  With it the studies' error norms without an analytic solution are
 * product norms of (reference solution - prolonged solution) on the reference level (test/linearelliptic.hh:205-214,
 * hdd_product_apply2 with "l2" / "h1_semi" / "elliptic").  HDD_ERR_INDEX_OUT_OF_RANGE for a father id outside the
 * coarse grid. */
int hdd_prolong(hdd_swipdg* coarse, const double* u_coarse_host, hdd_swipdg* fine, const int32_t* father_host,
                double* u_fine_host);

/* ---- BlockSWIPDG views (discretizations/block-swipdg.hh:553-690) --------------------------------------- */
int hdd_num_subdomains(const hdd_swipdg* h, int* n);
int hdd_subdomain_offsets(const hdd_swipdg* h, const int64_t** offsets_host); /* n+1 DoF offsets, mapToGlobal(ss,0) */
int hdd_neighbouring_subdomains(const hdd_swipdg* h, int ss, const int32_t** neighbours_host, int* n);
typedef struct hdd_csr {
  int64_t n_rows, n_cols, nnz;
  int64_t* rowptr;
  int32_t* col;
  double* val;
} hdd_csr;
/* get_local_operator(ss) (nn == ss) / get_coupling_operator(ss, nn): the (ss, nn) block of affine part q
 * (q = -1: affine part) with subdomain-local indices; host copy, release with hdd_csr_free. */
int hdd_block_extract(hdd_swipdg* h, int ss, int nn, int q, hdd_csr* out);
int hdd_csr_free(hdd_csr* m);

/* ---- estimators (estimators/swipdg.hh:824-985, estimators/block-swipdg.hh:1076-1265) ------------------- */
typedef struct hdd_parameters { /* the ParametersMapType keys of estimators/block-swipdg.hh:756-765 */
  const double* mu;
  const double* mu_hat;
  const double* mu_bar;
  const double* parameter_range_min;
  const double* parameter_range_max;
  int mu_size;
} hdd_parameters;

/* available(): "eta_NC_ESV2007", "eta_R_ESV2007", "eta_R_ESV2007_*", "eta_DF_ESV2007", "eta_ESV2007",
 * "eta_ESV2007_alt", "eta_NC_OS2014", "eta_R_OS2014", "eta_R_OS2014_*", "eta_DF_OS2014", "eta_DF_OS2014_*",
 * "eta_OS2014", "eta_OS2014_*".  Simplex grids only, like the reference (estimators/swipdg.hh:71). */
int hdd_estimators_available(const hdd_swipdg* h, const char* const** types, int* n_types);
/* estimate(space, vector, problem, type[, parameters]) -> eta;  u_host = NULL uses the last solution.
 * local_host (nullable): estimate_local(): n_cells (ESV2007 types) or n_subdomains (OS2014 types) entries. */
int hdd_estimate(hdd_swipdg* h, const char* type, const double* u_host, const hdd_parameters* parameters,
                 double* eta, double* local_host);
/* all squared per-cell indicators of one pass, for tests: out[8][n_owned] = nc2,res2,r2,df2,dfstar2,rstar2,amin,resstar2 */
int hdd_indicators(hdd_swipdg* h, const double* u_host, const hdd_parameters* parameters, double* out_host);

/* ---- multi GPU: one process per GPU ------------------------------------------------------------------------ */
/* NCCL plumbing: rank 0 calls hdd_comm_unique_id, the 128-byte id is broadcast by the host program
 * (torch.distributed), every rank creates ONE communicator per process with hdd_comm_create and attaches it to each
 * mesh whose owned range is a proper slab (hdd_mesh_attach_comm builds the halo-exchange plan).  NCCL carries only the
 * coupling-face halo exchange of the CG direction and the dot-product all-reduces.  All ranks must attach / solve /
 * estimate collectively. */
typedef struct hdd_comm hdd_comm;
int hdd_comm_unique_id(void* id128);
int hdd_comm_create(const void* id128, int rank, int world_size, int device, hdd_comm** out);
int hdd_comm_destroy(hdd_comm* comm);
int hdd_mesh_attach_comm(hdd_mesh* mesh, hdd_comm* comm);
/* The host-side partition plan hdd_mesh_create / hdd_comm_init build for `rank`, without touching a device (used by
 * the CPU tests of the N > 1 path and by hosts that want to inspect the decomposition): ranks own the consecutive
 * cell ranges rank_cell_offsets[r] .. rank_cell_offsets[r+1] (world_size+1 entries, whole subdomains).
 *   halo_cells   sorted global ids of every non-owned cell sharing a vertex with an owned cell (malloc'ed)
 *   send_cells   owned cells (global ids, sorted) whose DoFs peer r keeps in its halo, CSR by peer through
 *                send_offsets[world_size+1] (caller provided); equals peer r's halo cells owned by `rank`
 * Release both arrays with hdd_free. */
int hdd_partition_plan(int kind, int64_t n_cells, int64_t n_verts, const int32_t* cell_verts, int world_size,
                       const int64_t* rank_cell_offsets, int rank, int32_t** halo_cells, int64_t* n_halo,
                       int32_t** send_cells, int64_t* send_offsets);
/* The same plan computed the way hdd_mesh_create does it on N > 1 ranks: from the owned side only, walking face neighbours
 * across the partition faces (work proportional to the partition boundary, no sweep over the other ranks' cells); needs
 * the cell -> neighbour array.  Must equal hdd_partition_plan (tests/test_multi_gloo.py). */
int hdd_partition_plan_local(int kind, int64_t n_cells, const int32_t* cell_verts, const int32_t* cell_neigh, int world_size,
                             const int64_t* rank_cell_offsets, int rank, int32_t** halo_cells, int64_t* n_halo,
                             int32_t** send_cells, int64_t* send_offsets);
int hdd_free(void* p);
/* Entry points for tests (host arithmetic, the preconditioners' intermediate results) are in hdd_b200_testing.h. */

/* ---- measurement ------------------------------------------------------------------------------------------------ */
/* Times `reps` back-to-back launches of one hot kernel on the handle's stream with CUDA events (after 3 warm-up
 * launches) and returns the average launch duration: which = 0 the CG SpMV kernel (q = A p with the fused p.Ap
 * partial dot), 1 the fused CG update kernel, 2 the CG direction kernel, 3 the system-matrix assembly kernel of the
 * first affine part; 4 the device part of one estimator evaluation (Oswald vertex means, the per-cell indicator kernel
 * and the segmented reduction of its nine rows: the reference's four walks, estimators/swipdg.hh:668-687) on the vector
 * of the last hdd_estimate / hdd_indicators with default parameters; 5 the indicator kernel alone.  0-2 need a previous
 * hdd_solve (CG workspace), 4-5 a previous hdd_estimate.  Used by bench.py for the roofline numbers. */
int hdd_profile_kernel(hdd_swipdg* h, int which, int reps, double* avg_seconds);
/* algorithmic HBM bytes of one launch of that kernel (DESIGN.md "Kernels and rooflines") */
int hdd_kernel_bytes(hdd_swipdg* h, int which, double* bytes);

/* ParameterFunctional / Expression evaluation on the host (no device needed): value of `expression` in the vector
 * variable `variable` ("x" or "mu") at `values[0..n)`.  HDD_ERR_WRONG_INPUT on a syntax error. */
int hdd_expression_evaluate(const char* expression, const char* variable, const double* values, int n, double* out);

/* ---- counters --------------------------------------------------------------------------------------------------- */
/* number of kernels this library launched since process start (bench.py's gpu_launches) */
int64_t hdd_kernel_launches(void);
/* bytes this library copied from host to device memory since process start (bench.py's e2e.h2d_bytes_per_step) */
int64_t hdd_h2d_bytes(void);

#ifdef __cplusplus
}
#endif
#endif /* HDD_B200_H */
