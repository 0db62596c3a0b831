/*
 * hdd_b200_testing.h - entry points of libhdd_b200 that exist for tests: host arithmetic the CPU tests check without a
 * device, and views into the solvers' intermediate results that the GPU tests compare with a plain float64 restatement
 * (tests/mg_reference.py).  A drop-in host of the reference needs none of them; conventions as in hdd_b200.h.
 */
#ifndef HDD_B200_TESTING_H
#define HDD_B200_TESTING_H

#include "hdd_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Host arithmetic of the strip-distributed multigrid preconditioner ("cg.mg" on N GPUs, DESIGN.md 7): the inclusive
 * vertex-row ranges the sweeps of the n_dist finest vertex levels run on for the rank owning the cell rows [c0, c1) of an
 * ny-row structured grid.  out[8 l + k], k = 0..7: pre_lo, pre_hi (pre-smoothing), b_lo, b_hi (right-hand side), up_lo,
 * up_hi (post-smoothing), pro_lo, pro_hi (prolongation) of level l; out[8 n_dist + {0,1,2}]: first and last own row of the
 * first replicated level, and the number of level-0 rows received from each neighbour.  No device needed. */
int hdd_mg_strip_plan(int ny, int c0, int c1, int n_dist, int* out);
/* The branch-free cosine the estimator kernel evaluates trigonometric data functions with (csrc/expr.hpp: fast_cos, valid
 * for |x| <= 1e5), run on the host: out[i] = fast_cos(x[i]).  No device needed. */
int hdd_fast_cos(const double* x, int64_t n, double* out);
/* Whether the kernels would evaluate the Expression `expression` (variable "x") as a product of at most two cosines of
 * affine arguments (csrc/expr.hpp: TrigProduct), and with which numbers: out[7] = c, a0, b0, d0, a1, b1, d1 of
 * c cos(a0 x[0] + b0 x[1] + d0) cos(a1 x[0] + b1 x[1] + d1); *valid = 0 if the expression has another shape (it is then
 * evaluated by the general path).  No device needed. */
int hdd_trig_product(const char* expression, double* out, int* valid);

/* z = M^-1 r: one application of the preconditioner of solver type `type` (names and aliases as hdd_solve) for the
 * operator frozen at mu, through hdd_solve's own set-up and CG initialisation (z is the first search direction of a
 * solve whose right-hand side is r).  r_host, z_host: n_owned.  rz (nullable): r.z as the solver's fused reduction
 * computed it.  vertex_host (nullable; cg.mg / cg.mg2 only): the V-cycle results on the finest vertex level,
 * n_hier (nx+1)(ny+1) doubles - cg.mg on cubes: V(P^T r), V_C(C P^T r); on lattice simplices: V(P^T r);
 * cg.mg2: V_P(P^T r), V_H(H^T r).  Leaves the solution, the rhs and hdd_solve's cached CUDA graphs untouched.
 * One GPU only; HDD_ERR_NOT_IMPLEMENTED on N GPUs and for purely Neumann problems. */
int hdd_precondition(hdd_swipdg* h, const char* type, const double* mu, int mu_size, const double* r_host,
                     double* z_host, double* rz, double* vertex_host);

/* The 9-point operator of multigrid level `level`, hierarchy `hier`, as the last cg.mg / cg.mg2 set-up left it:
 * nx, ny of the level's vertex grid; S_host (nullable) 9 (nx+1)(ny+1) doubles, S[e nv + v] = coupling of
 * v = (ix, iy) to (ix+dx, iy+dy), e = 3 (dy+1) + dx + 1.  HDD_ERR_WRONG_INPUT past the coarsest level, for a
 * hierarchy that does not exist, and for level 0 of cg.mg's twisted hierarchy (C A_c C is not stored). */
int hdd_mg_level_operator(const hdd_swipdg* h, int level, int hier, int* nx, int* ny, double* S_host);

#ifdef __cplusplus
}
#endif
#endif /* HDD_B200_TESTING_H */
