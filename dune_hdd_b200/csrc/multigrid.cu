// "cg.mg": CG preconditioned by a two-level method for the SWIPDG matrix on logically structured Q1 grids.
//
//   M^-1 r = D_blk^-1 r  +  P V(P^T r)  +  P C V_C(C P^T r)
//
// D_blk   the 4 x 4 cell blocks of A (block Jacobi, the DG-level smoother),
// P       the injection of the conforming Q1 space into the DG space (DG DoF (T, i) = value at vertex i of T); the
//         auxiliary operator A_c = P^T A P is a 9-point vertex stencil (for continuous functions every inner-face jump
//         vanishes, what remains is the volume term and the Dirichlet-face terms),
// V       one geometric multigrid V(1,1)-cycle for A_c on the (nx+1) x (ny+1) vertex grid: damped Jacobi, bilinear
//         interpolation, full weighting, Galerkin coarse operators, dense inverse on the coarsest grid,
// C       the checkerboard sign (-1)^(ix+iy).  The reference under-integrates the Q1 volume term with the midpoint rule
//         (SURVEY 0.4), which makes the element hourglass mode energy-free: A_c has a second family of low-energy modes,
//         checkerboard x smooth, invisible to standard coarse grids.  The twisted hierarchy V_C built from C A_c C
//         removes exactly that family (measured: CG iterations 188 -> 42 at 128^2, flat in h; see DESIGN.md).
//
// The reference's default solver is BiCGSTAB with an algebraic-multigrid / ILU preconditioner
// (Stuff::LA::Solver defaults, discretizations/base.hh:314-322, SURVEY 0.5); this is the same idea specialised to the
// structured grids of BASELINE configs 2 and 5.  Everything is additive and symmetric, so CG stays applicable; all
// reductions are deterministic.
//
// Multi GPU: the DG level (SpMV, block Jacobi, restriction, prolongation) is distributed like the rest of the solve.
// The vertex-level operators are replicated (one all-reduce per solve makes the level-0 stencil global); when the ranks'
// cells are full-width bands of rows stacked in rank order (the slabs bench.py deals out), the vectors of the two finest
// vertex levels are swept in row strips with one halo row exchanged per sweep (grouped ncclSend/ncclRecv with the rank
// below / above), the level-2 right-hand side is summed over the ranks and levels >= 2 run replicated.  Otherwise the
// whole V-cycle runs replicated on the all-reduced restricted residual.
//
// "cg.mg2": the same machinery for polOrder 2 on structured Q2 grids,
//
//   M^-1 r = D_9^-1 r  +  P V_P(P^T r)  +  H V_H(H^T r)
//
// with P the bilinear interpolation of the conforming Q1 space into Q2-DG and H the hourglass family of the Q2 volume
// term (see k_vertex_galerkin_q2).  A_P and A_H are two independent 9-point vertex operators: the two hierarchies of
// MgState (MgKind::mg2), each with a level-0 operator of its own.  On N GPUs the vertex levels always run replicated.
//
// "cg.mg2.simplex": polOrder 2 on lattice-structured triangle grids,
//
//   M^-1 r = D_6^-1 r  +  P V(P^T r)
//
// with P the interpolation of the conforming P1 space on the vertex lattice into P2-DG (see k_vertex_galerkin_p2).  The P2
// volume rule is exact, so there is no hourglass family: one hierarchy, the vertex levels of the P1 lattice path of
// "cg.mg", and only the DG level is new.  On N GPUs the vertex levels run replicated, as for "cg.mg2".
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <ctime>

#include "handles.hpp"
#include "reduce.cuh"

namespace hdd {

namespace {

constexpr int kMgThreads = 256;
constexpr int kMaxCoarse = 400;   // dense coarsest solve up to this many vertices
constexpr double kOmega = 0.8;    // Jacobi damping on the vertex levels

inline int blocks_for(int64_t n) { return int((n + kMgThreads - 1) / kMgThreads); }

// The vertices (linear index range = whole grid rows) a kernel launch works on: the whole level, or - for the levels
// that are distributed over the GPUs - the row strip this rank owns.
struct Rows {
  int64_t beg, cnt;
};

__device__ __forceinline__ void load_neigh4(const int32_t* neigh, int k, int* nb) {
  const int4 v = __ldg(reinterpret_cast<const int4*>(neigh) + k);
  nb[0] = v.x; nb[1] = v.y; nb[2] = v.z; nb[3] = v.w;
}

// ---- structure detection -------------------------------------------------------------------------------------
// cells: vertices must be (v0, v0+1, v0+nx1, v0+nx1+1); records v0 per cell and the map lexicographic cell -> cell
__global__ void k_struct_cells(const int32_t* __restrict__ cv, int32_t n_cells, int nx, int ny, int32_t* __restrict__ cell_v0,
                               int32_t* __restrict__ lex_cell, int32_t* flag) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;  // local cell id
  if (c >= n_cells) return;
  const int4 v = __ldg(reinterpret_cast<const int4*>(cv) + c);
  const int nx1 = nx + 1;
  const int cx = v.x % nx1, cy = v.x / nx1;
  if (v.x < 0 || cx >= nx || cy >= ny || v.y != v.x + 1 || v.z != v.x + nx1 || v.w != v.x + nx1 + 1) {
    atomicOr(flag, 1);
    return;
  }
  cell_v0[c] = v.x;
  lex_cell[cx + nx * cy] = c;
}

// triangles: the three vertices must be pairwise lattice neighbours (index distance <= 1 in both directions)
__global__ void k_struct_triangles(const int32_t* __restrict__ cv, int32_t n_cells, int nx1, int64_t n_verts, int32_t* flag) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  int vx[3], vy[3];
  for (int i = 0; i < 3; ++i) {
    const int v = cv[size_t(3) * c + i];
    if (v < 0 || v >= n_verts) { atomicOr(flag, 1); return; }
    vx[i] = v % nx1;
    vy[i] = v / nx1;
  }
  for (int i = 0; i < 3; ++i) {
    const int j = (i + 1) % 3;
    if (abs(vx[i] - vx[j]) > 1 || abs(vy[i] - vy[j]) > 1) atomicOr(flag, 1);
  }
}

// vertices [v0, v0 + count): tensor-product coordinates, checked against the one-dimensional coordinate tables
__global__ void k_struct_verts(const double* __restrict__ xy /* indexed by global vertex id */, int64_t v0, int64_t count, int nx,
                               const double* __restrict__ xs, const double* __restrict__ ys, int32_t* flag) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const int64_t v = v0 + t;
  const int nx1 = nx + 1;
  const double2 p = __ldg(reinterpret_cast<const double2*>(xy) + v);
  if (p.x != __ldg(xs + v % nx1) || p.y != __ldg(ys + v / nx1)) atomicOr(flag, 2);
}

// one-dimensional geometry of the tensor grid: {x0, hx, 1/hx, -} per column followed by {y0, hy, 1/hy, -} per row
// (the reciprocals save the assembly kernel six of its ten fp64 divisions per cell)
__global__ void k_struct_geo(const double* __restrict__ xs, const double* __restrict__ ys, int nx, int ny, double* __restrict__ tgeo) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nx + ny) return;
  double4* out = reinterpret_cast<double4*>(tgeo);
  if (t < nx) {
    const double x0 = xs[t], x1 = xs[t + 1];
    out[t] = make_double4(x0, x1 - x0, 1.0 / (x1 - x0), 0.0);
  } else {
    const int r = t - nx;
    const double y0 = ys[r], y1 = ys[r + 1];
    out[t] = make_double4(y0, y1 - y0, 1.0 / (y1 - y0), 0.0);
  }
}

// ---- level-0 operator: A_c = P^T A P gathered per vertex (no atomics) ------------------------------------------
// S[e][v], e = (dy+1)*3 + (dx+1): coupling of vertex v = (ix, iy) to vertex (ix+dx, iy+dy).  Entries of P^T A P at
// index distance 2 cancel analytically (inner-face jumps of continuous functions) and are dropped.
__global__ void __launch_bounds__(kMgThreads)
    k_vertex_galerkin(MeshView m, const double* __restrict__ vals, const int32_t* __restrict__ cell_v0,
                      const int32_t* __restrict__ lex_cell, int nx, int ny, Rows rg, double* __restrict__ S) {
  const int64_t nv = int64_t(nx + 1) * (ny + 1);
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const int64_t v = rg.beg + tid;
  const int nx1 = nx + 1;
  const int ix = int(v % nx1), iy = int(v / nx1);
  double acc[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) acc[e] = 0.0;
#pragma unroll
  for (int b = 0; b < 2; ++b)
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int cx = ix - 1 + a, cy = iy - 1 + b;
      if (cx < 0 || cy < 0 || cx >= nx || cy >= ny) continue;
      const int c = __ldg(lex_cell + cx + nx * cy);  // local cell id, -1 = not on this rank
      const int k = c - m.own0;
      if (c < 0 || k < 0 || k >= m.n_own) continue;  // rows of cells owned elsewhere are added by the all-reduce
      const int i = (1 - a) + 2 * (1 - b);  // local index of v in that cell
      int nb[4];
      load_neigh4(m.neigh, k, nb);
      const int nblk = block_count<4>(nb);
      const double* row = vals + __ldg(m.blk_start + k) * 16 + int64_t(i) * nblk * 4;
#pragma unroll
      for (int t = 0; t < 5; ++t) {
        const int cell = t == 0 ? c : nb[t - 1];
        if (cell < 0) continue;
        const int slot = block_slot<4>(c, nb, cell);
        const int v0 = __ldg(cell_v0 + cell);
        const int jx = v0 % nx1 - ix, jy = v0 / nx1 - iy;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int dx = jx + (j & 1), dy = jy + (j >> 1);
          if (dx < -1 || dx > 1 || dy < -1 || dy > 1) continue;
          acc[(dy + 1) * 3 + dx + 1] += __ldg(row + slot * 4 + j);
        }
      }
    }
#pragma unroll
  for (int e = 0; e < 9; ++e) S[e * nv + v] = acc[e];
}

// b1 = C b0 after the all-reduce of b0 (multi GPU)
__global__ void k_twist_vector(const int* done, const double* __restrict__ b0, int nx, Rows rg, double* __restrict__ b1) {
  if (done && *done) return;
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const int64_t v = rg.beg + tid;
  const int nx1 = nx + 1;
  b1[v] = ((int(v % nx1) + int(v / nx1)) & 1) ? -b0[v] : b0[v];
}

// ---- Galerkin coarse operator with bilinear interpolation: 9-point -> 9-point ---------------------------------
// Coarse vertices of the row range rg (reads the fine operator on the fine rows 2 I - 1 .. 2 I + 1 only).  blockIdx.y
// picks the hierarchy: fine / coarse operators hf / hc entries apart; twist_h1: the fine operator of hierarchy 1 is
// C A C, read from the arrays of A (level 0 -> 1).
__global__ void __launch_bounds__(kMgThreads)
    k_rap(const double* __restrict__ Sf, int64_t hf, int nxf, int nyf, int twist_h1, Rows rg, double* __restrict__ Sc, int64_t hc) {
  const int nxc = nxf / 2, nyc = nyf / 2;
  const int64_t nvc = int64_t(nxc + 1) * (nyc + 1), nvf = int64_t(nxf + 1) * (nyf + 1);
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const int twist = twist_h1 && blockIdx.y == 1;
  Sf += int64_t(blockIdx.y) * hf;
  Sc += int64_t(blockIdx.y) * hc;
  const int64_t I = rg.beg + tid;
  const int IX = int(I % (nxc + 1)), IY = int(I / (nxc + 1));
  double acc[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) acc[e] = 0.0;
  for (int dy = -1; dy <= 1; ++dy)
    for (int dx = -1; dx <= 1; ++dx) {
      const int fx = 2 * IX + dx, fy = 2 * IY + dy;
      if (fx < 0 || fy < 0 || fx > nxf || fy > nyf) continue;
      const double wd = (dx == 0 ? 1.0 : 0.5) * (dy == 0 ? 1.0 : 0.5);
      const int64_t i = fx + int64_t(nxf + 1) * fy;
      for (int ey = -1; ey <= 1; ++ey)
        for (int ex = -1; ex <= 1; ++ex) {
          const int jx = fx + ex, jy = fy + ey;
          if (jx < 0 || jy < 0 || jx > nxf || jy > nyf) continue;
          double s = wd * __ldg(Sf + ((ey + 1) * 3 + ex + 1) * nvf + i);
          if (twist && ((ex + ey) & 1)) s = -s;  // fine operator C A C, read from the arrays of A
          // coarse vertices J = I + D whose interpolation stencil touches j: |j - 2J| <= 1
#pragma unroll
          for (int Dy = -1; Dy <= 1; ++Dy) {
            const int py = dy + ey - 2 * Dy;
            if (py < -1 || py > 1 || IY + Dy < 0 || IY + Dy > nyc) continue;
#pragma unroll
            for (int Dx = -1; Dx <= 1; ++Dx) {
              const int px = dx + ex - 2 * Dx;
              if (px < -1 || px > 1 || IX + Dx < 0 || IX + Dx > nxc) continue;
              acc[(Dy + 1) * 3 + Dx + 1] += s * (px == 0 ? 1.0 : 0.5) * (py == 0 ? 1.0 : 0.5);
            }
          }
        }
    }
#pragma unroll
  for (int e = 0; e < 9; ++e) Sc[e * nvc + I] = acc[e];
}

// ---- V-cycle kernels.  done: convergence latch of the CG iteration that owns this application (see k_cg_*) ----------
// On levels >= 1 the two hierarchies (plain and twisted) are swept by the same launch: blockIdx.y picks the hierarchy,
// its operator sits 9 nv and its vectors nv entries behind those of the plain one.
// pre-smoothing from a zero guess, x = w D^-1 b, fused with the residual r = b - A x
__global__ void __launch_bounds__(kMgThreads)
    k_mg_pre(const int* done, const double* __restrict__ S, const double* __restrict__ dinv, int nx, int ny, Rows rg,
             const double* __restrict__ b, double* __restrict__ x, double* __restrict__ r) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const int64_t hv = int64_t(blockIdx.y) * nv;
  S += 9 * hv; dinv += hv; b += hv; x += hv; r += hv;
  const int64_t i = rg.beg + tid;
  const int ix = int(i % nx1), iy = int(i / nx1);
  double ax = 0.0;
#pragma unroll
  for (int ey = -1; ey <= 1; ++ey)
#pragma unroll
    for (int ex = -1; ex <= 1; ++ex) {
      const int jx = ix + ex, jy = iy + ey;
      if (jx < 0 || jy < 0 || jx > nx || jy > ny) continue;
      const int64_t j = i + ex + int64_t(ey) * nx1;
      const double xj = __ldg(dinv + j) * __ldg(b + j);  // dinv = w / diagonal: no division in the sweep
      ax = fma(__ldg(S + ((ey + 1) * 3 + ex + 1) * nv + i), xj, ax);
      if (ex == 0 && ey == 0) x[i] = xj;
    }
  r[i] = b[i] - ax;
}

// full weighting: b_H = P^T r (both hierarchies)
__global__ void __launch_bounds__(kMgThreads)
    k_mg_restrict(const int* done, const double* __restrict__ r, int nxf, int nyf, Rows rg /* coarse */, double* __restrict__ bc) {
  if (done && *done) return;
  const int nxc = nxf / 2, nyc = nyf / 2;
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  r += int64_t(blockIdx.y) * (int64_t(nxf + 1) * (nyf + 1));
  bc += int64_t(blockIdx.y) * (int64_t(nxc + 1) * (nyc + 1));
  const int64_t I = rg.beg + tid;
  const int IX = int(I % (nxc + 1)), IY = int(I / (nxc + 1));
  double s = 0.0;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int fx = 2 * IX + dx, fy = 2 * IY + dy;
      if (fx < 0 || fy < 0 || fx > nxf || fy > nyf) continue;
      s = fma((dx == 0 ? 1.0 : 0.5) * (dy == 0 ? 1.0 : 0.5), __ldg(r + fx + int64_t(nxf + 1) * fy), s);
    }
  bc[I] = s;
}

// value of the bilinear interpolant P x_H at the fine vertex (fx, fy)
__device__ __forceinline__ double mg_interp(const double* __restrict__ xc, int nxc1, int fx, int fy) {
  const int ox = fx & 1, oy = fy & 1;
  const int64_t I = (fx >> 1) + int64_t(nxc1) * (fy >> 1);
  double v = __ldg(xc + I);
  if (ox) v += __ldg(xc + I + 1);
  if (oy) {
    v += __ldg(xc + I + nxc1);
    if (ox) v += __ldg(xc + I + nxc1 + 1);
  }
  return v * (ox ? 0.5 : 1.0) * (oy ? 0.5 : 1.0);
}

// x += P x_H (bilinear interpolation), both hierarchies
__global__ void __launch_bounds__(kMgThreads)
    k_mg_prolong_add(const int* done, const double* __restrict__ xc, int nxf, int nyf, Rows rg /* fine */, double* __restrict__ x) {
  if (done && *done) return;
  const int nxc = nxf / 2, nyc = nyf / 2;
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  x += int64_t(blockIdx.y) * (int64_t(nxf + 1) * (nyf + 1));
  xc += int64_t(blockIdx.y) * (int64_t(nxc + 1) * (nyc + 1));
  const int64_t i = rg.beg + tid;
  x[i] += mg_interp(xc, nxc + 1, int(i % (nxf + 1)), int(i / (nxf + 1)));
}

// post-smoothing: y = x + w D^-1 (b - A x), both hierarchies
__global__ void __launch_bounds__(kMgThreads)
    k_mg_post(const int* done, const double* __restrict__ S, const double* __restrict__ dinv, int nx, int ny, Rows rg,
              const double* __restrict__ b, const double* __restrict__ x, double* __restrict__ y) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const int64_t hv = int64_t(blockIdx.y) * nv;
  S += 9 * hv; dinv += hv; b += hv; x += hv; y += hv;
  const int64_t i = rg.beg + tid;
  const int ix = int(i % nx1), iy = int(i / nx1);
  double ax = 0.0;
#pragma unroll
  for (int ey = -1; ey <= 1; ++ey)
#pragma unroll
    for (int ex = -1; ex <= 1; ++ex) {
      const int jx = ix + ex, jy = iy + ey;
      if (jx < 0 || jy < 0 || jx > nx || jy > ny) continue;
      ax = fma(__ldg(S + ((ey + 1) * 3 + ex + 1) * nv + i), __ldg(x + i + ex + int64_t(ey) * nx1), ax);
    }
  y[i] = fma(__ldg(dinv + i), b[i] - ax, x[i]);
}

// prolongation and post-smoothing in one sweep for the small levels, where a launch costs more than the arithmetic:
// y = xp + w D^-1 (b - A xp) with xp = x + P x_H formed on the fly at the nine stencil points (same operations, same
// results as k_mg_prolong_add followed by k_mg_post)
__global__ void __launch_bounds__(kMgThreads)
    k_mg_up(const int* done, const double* __restrict__ S, const double* __restrict__ dinv, int nx, int ny, Rows rg,
            const double* __restrict__ b, const double* __restrict__ x, const double* __restrict__ xc, double* __restrict__ y) {
  if (done && *done) return;
  const int nx1 = nx + 1, nxc1 = nx / 2 + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const int64_t hv = int64_t(blockIdx.y) * nv;
  S += 9 * hv; dinv += hv; b += hv; x += hv; y += hv;
  xc += int64_t(blockIdx.y) * (int64_t(nxc1) * (ny / 2 + 1));
  const int64_t i = rg.beg + tid;
  const int ix = int(i % nx1), iy = int(i / nx1);
  double ax = 0.0, xi = 0.0;
#pragma unroll
  for (int ey = -1; ey <= 1; ++ey)
#pragma unroll
    for (int ex = -1; ex <= 1; ++ex) {
      const int jx = ix + ex, jy = iy + ey;
      if (jx < 0 || jy < 0 || jx > nx || jy > ny) continue;
      const double xp = __ldg(x + i + ex + int64_t(ey) * nx1) + mg_interp(xc, nxc1, jx, jy);
      ax = fma(__ldg(S + ((ey + 1) * 3 + ex + 1) * nv + i), xp, ax);
      if (ex == 0 && ey == 0) xi = xp;
    }
  y[i] = fma(__ldg(dinv + i), b[i] - ax, xi);
}

// Level 0, both hierarchies in one sweep: C A_c C differs from A_c only by the sign of the edge-neighbour entries
// (e odd), so the nine coefficient arrays - three quarters of the bytes of a smoothing sweep - are read once for
// the plain and the twisted hierarchy.  The vectors of the twisted hierarchy sit nv entries behind the plain ones.
__global__ void __launch_bounds__(kMgThreads)
    k_mg_pre2(const int* done, const double* __restrict__ S, const double* __restrict__ dinv, int nx, int ny, Rows rg,
              const double* __restrict__ b0, double* __restrict__ x0, double* __restrict__ r0) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const double* b1 = b0 + nv;
  double* x1 = x0 + nv;
  double* r1 = r0 + nv;
  const int64_t i = rg.beg + tid;
  const int ix = int(i % nx1), iy = int(i / nx1);
  double a0 = 0.0, a1 = 0.0;
#pragma unroll
  for (int ey = -1; ey <= 1; ++ey)
#pragma unroll
    for (int ex = -1; ex <= 1; ++ex) {
      const int jx = ix + ex, jy = iy + ey;
      if (jx < 0 || jy < 0 || jx > nx || jy > ny) continue;
      const int64_t j = i + ex + int64_t(ey) * nx1;
      const double dj = __ldg(dinv + j);
      const double xj0 = dj * __ldg(b0 + j), xj1 = dj * __ldg(b1 + j);
      const double se = __ldg(S + ((ey + 1) * 3 + ex + 1) * nv + i);
      a0 = fma(se, xj0, a0);
      a1 = fma(((ex + ey) & 1) ? -se : se, xj1, a1);
      if (ex == 0 && ey == 0) { x0[i] = xj0; x1[i] = xj1; }
    }
  r0[i] = b0[i] - a0;
  r1[i] = b1[i] - a1;
}

__global__ void __launch_bounds__(kMgThreads)
    k_mg_post2(const int* done, const double* __restrict__ S, const double* __restrict__ dinv, int nx, int ny, Rows rg,
               const double* __restrict__ b0, const double* __restrict__ x0, double* __restrict__ y0) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const double* b1 = b0 + nv;
  const double* x1 = x0 + nv;
  double* y1 = y0 + nv;
  const int64_t i = rg.beg + tid;
  const int ix = int(i % nx1), iy = int(i / nx1);
  double a0 = 0.0, a1 = 0.0;
#pragma unroll
  for (int ey = -1; ey <= 1; ++ey)
#pragma unroll
    for (int ex = -1; ex <= 1; ++ex) {
      const int jx = ix + ex, jy = iy + ey;
      if (jx < 0 || jy < 0 || jx > nx || jy > ny) continue;
      const int64_t j = i + ex + int64_t(ey) * nx1;
      const double se = __ldg(S + ((ey + 1) * 3 + ex + 1) * nv + i);
      a0 = fma(se, __ldg(x0 + j), a0);
      a1 = fma(((ex + ey) & 1) ? -se : se, __ldg(x1 + j), a1);
    }
  const double d = __ldg(dinv + i);
  y0[i] = fma(d, b0[i] - a0, x0[i]);
  y1[i] = fma(d, b1[i] - a1, x1[i]);
}

// dinv = w / diagonal of the level operator (both hierarchies)
__global__ void k_mg_dinv(const double* __restrict__ S, int64_t nv, Rows rg, double* __restrict__ dinv) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t hv = int64_t(blockIdx.y) * nv;
  if (t < rg.cnt) dinv[hv + rg.beg + t] = kOmega / S[9 * hv + 4 * nv + rg.beg + t];
}

// coarsest grid: x = A^-1 b with the dense inverse, one warp per row (lanes along the row: coalesced, 9 products per lane
// at n = 289, then a shuffle reduction - one thread per row was a chain of n dependent loads, 50 us).  Both hierarchies.
__global__ void k_mg_dense(const int* done, const double* __restrict__ Ainv, int n, const double* __restrict__ b,
                           double* __restrict__ x) {
  if (done && *done) return;
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  Ainv += size_t(blockIdx.y) * n * n;
  b += size_t(blockIdx.y) * n;
  x += size_t(blockIdx.y) * n;
  double s = 0.0;
  for (int j = lane; j < n; j += 32) s = fma(__ldg(Ainv + size_t(i) * n + j), __ldg(b + j), s);
  s = warp_sum(s);
  if (lane == 0) x[i] = s;
}

// Dense inverse of the coarsest operator (s.p.d., n <= kMaxCoarse) on the device: Gauss-Jordan without pivoting, one CTA per
// hierarchy, [A | inv] in global memory (L2 resident).  Per pivot: the pivot column is saved in shared memory, then every
// warp updates the rows that have a non-zero there (a 9-point operator: ~2 (nx + 2) rows) with its lanes along the row.
// The host version of this loop took 7-15 ms per hierarchy and solve - at 8 GPUs a quarter of the whole solve.
// flag |= 1 if a pivot is not positive.  twist: hierarchy 1 reads C A C from the arrays of A (single-level case).
__global__ void __launch_bounds__(1024)
    k_dense_inverse(const double* __restrict__ S, int64_t hs /* operator stride between the hierarchies */, int nx, int ny,
                    int twist_h1, double* __restrict__ work, double* __restrict__ inv, int* flag) {
  __shared__ double col[kMaxCoarse];
  __shared__ double pivot_inv;
  const int nx1 = nx + 1, n = nx1 * (ny + 1);
  const int h = blockIdx.x;
  const bool twist = twist_h1 && h == 1;
  S += int64_t(h) * hs;
  double* A = work + size_t(h) * n * n;
  double* I = inv + size_t(h) * n * n;
  for (int t = threadIdx.x; t < n * n; t += blockDim.x) {
    const int i = t / n, j = t - i * n;
    const int ix = i % nx1, iy = i / nx1, jx = j % nx1, jy = j / nx1;
    const int ex = jx - ix, ey = jy - iy;
    double a = 0.0;
    if (ex >= -1 && ex <= 1 && ey >= -1 && ey <= 1) {
      a = S[int64_t((ey + 1) * 3 + ex + 1) * n + i];
      if (twist && ((ex + ey) & 1)) a = -a;
    }
    A[t] = a;
    I[t] = i == j ? 1.0 : 0.0;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, n_warps = blockDim.x >> 5;
  for (int c = 0; c < n; ++c) {
    if (threadIdx.x == 0) {
      const double piv = A[size_t(c) * n + c];
      if (!(piv > 0.0)) atomicOr(flag, 1);
      pivot_inv = 1.0 / piv;
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) col[i] = i == c ? 0.0 : A[size_t(i) * n + c];
    __syncthreads();
    const double ip = pivot_inv;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      A[size_t(c) * n + j] *= ip;
      I[size_t(c) * n + j] *= ip;
    }
    __syncthreads();
    for (int i = warp; i < n; i += n_warps) {
      const double f = col[i];
      if (f == 0.0) continue;
      for (int j = lane; j < n; j += 32) {
        A[size_t(i) * n + j] = fma(-f, A[size_t(c) * n + j], A[size_t(i) * n + j]);
        I[size_t(i) * n + j] = fma(-f, I[size_t(c) * n + j], I[size_t(i) * n + j]);
      }
    }
    __syncthreads();
  }
}

// The same inverse through a banded Cholesky factorisation (the 9-point operator on an nx1-wide lattice has half bandwidth
// w = nx1 + 1): A = L L^T with L kept as a band in shared memory (n (w + 1) doubles: 44 KB for 17 x 17), then thread k solves
// L y = e_k, L^T x = y for column k of the inverse - n independent substitutions running in lockstep, the L entries broadcast
// from shared memory, y and x in the (L2-resident) work / inv arrays with coalesced rows.  O(n w^2 + n^2 w) operations instead
// of the O(n^3) of Gauss-Jordan, and two barriers per column instead of three plus a sweep over every row: ~0.2 ms instead of
// ~9 ms for the two 289 x 289 operators of the 4096^2 hierarchy (a fifth of the whole solve at 8 GPUs).
// One CTA per hierarchy, blockDim.x >= n.  flag |= 1 if a pivot is not positive.
__global__ void __launch_bounds__(512)
    k_dense_inverse_banded(const double* __restrict__ S, int64_t hs, int nx, int ny, int twist_h1, double* __restrict__ work,
                           double* __restrict__ inv, int* flag) {
  extern __shared__ __align__(16) double Lb[];  // Lb[i * (w + 1) + d] = L[i][i - d]
  __shared__ double piv;
  const int nx1 = nx + 1, n = nx1 * (ny + 1), w = nx1 + 1, ld = w + 1;
  const int h = blockIdx.x;
  const bool twist = twist_h1 && h == 1;
  S += int64_t(h) * hs;
  double* Y = work + size_t(h) * n * n;
  double* X = inv + size_t(h) * n * n;
  for (int t = threadIdx.x; t < n * ld; t += blockDim.x) {
    const int i = t / ld, d = t - i * ld, j = i - d;
    double a = 0.0;
    if (j >= 0) {
      const int ix = i % nx1, iy = i / nx1, jx = j % nx1, jy = j / nx1;
      const int ex = jx - ix, ey = jy - iy;
      if (ex >= -1 && ex <= 1 && ey >= -1 && ey <= 1) {
        a = S[int64_t((ey + 1) * 3 + ex + 1) * n + i];
        if (twist && ((ex + ey) & 1)) a = -a;
      }
    }
    Lb[t] = a;
  }
  __syncthreads();
  // left-looking banded Cholesky: thread t of the first w + 1 computes L[j + t][j]
  for (int j = 0; j < n; ++j) {
    const int t = threadIdx.x, i = j + t;
    double v = 0.0;
    if (t <= w && i < n) {
      v = Lb[i * ld + t];                          // A[i][j]
      for (int d = 1; d + t <= w && d <= j; ++d)   // k = j - d: L[i][k] = Lb[i][t + d], L[j][k] = Lb[j][d]
        v = fma(-Lb[i * ld + t + d], Lb[j * ld + d], v);
      if (t == 0) {
        if (!(v > 0.0)) atomicOr(flag, 1);
        piv = sqrt(v);
      }
    }
    __syncthreads();
    if (t <= w && i < n) Lb[i * ld + t] = t == 0 ? piv : v / piv;
    __syncthreads();
  }
  const int k = threadIdx.x;
  if (k >= n) return;
  // forward: L y = e_k (y_i = 0 for i < k)
  for (int i = 0; i < n; ++i) {
    double sacc = i == k ? 1.0 : 0.0;
    if (i > k) {
      const int dmax = min(w, i - k);
      for (int d = 1; d <= dmax; ++d) sacc = fma(-Lb[i * ld + d], Y[size_t(i - d) * n + k], sacc);
    }
    Y[size_t(i) * n + k] = i < k ? 0.0 : sacc / Lb[i * ld];
  }
  // backward: L^T x = y
  for (int i = n - 1; i >= 0; --i) {
    double sacc = Y[size_t(i) * n + k];
    const int dmax = min(w, n - 1 - i);
    for (int d = 1; d <= dmax; ++d) sacc = fma(-Lb[(i + d) * ld + d], X[size_t(i + d) * n + k], sacc);
    X[size_t(i) * n + k] = sacc / Lb[i * ld];
  }
}

// ---- DG level ---------------------------------------------------------------------------------------------------
// rc = P^T r (sum of the DG residual entries sitting on each vertex) and its checkerboard-signed copy
__global__ void __launch_bounds__(kMgThreads)
    k_dg_restrict(const int* done, const double* __restrict__ r, const int32_t* __restrict__ lex_cell, int own0,
                  int n_own, int nx, int ny, Rows rg, double* __restrict__ b0, double* __restrict__ b1) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= rg.cnt) return;
  const int64_t v = rg.beg + tid;
  const int ix = int(v % nx1), iy = int(v / nx1);
  double s = 0.0;
#pragma unroll
  for (int b = 0; b < 2; ++b)
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int cx = ix - 1 + a, cy = iy - 1 + b;
      if (cx < 0 || cy < 0 || cx >= nx || cy >= ny) continue;
      const int k = __ldg(lex_cell + cx + nx * cy) - own0;
      if (k < 0 || k >= n_own) continue;
      s += __ldg(r + size_t(4) * k + (1 - a) + 2 * (1 - b));
    }
  b0[v] = s;
  if (b1) b1[v] = ((ix + iy) & 1) ? -s : s;
}

// Strip-distributed application, after the exchange of the level-0 right-hand side: lo / up hold the g + 1 vertex rows
// [c0 - g, c0] of the rank below and [c1, c1 + g] of the rank above.  The shared rows c0 and c1 were summed over this
// rank's cells only - the neighbour's share is added (two summands: the order does not matter) - the other rows are
// copied, and the checkerboard-signed copy b1 = C b0 is written for the whole range [rows lo_row, hi_row].
__global__ void __launch_bounds__(kMgThreads)
    k_ghost_unpack_twist(const int* done, double* __restrict__ b0, double* __restrict__ b1, const double* __restrict__ lo,
                         const double* __restrict__ up, int nx, int c0, int c1, int g, int lo_row, int hi_row) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= int64_t(hi_row - lo_row + 1) * nx1) return;
  const int64_t v = int64_t(lo_row) * nx1 + tid;
  const int ix = int(v % nx1), iy = int(v / nx1);
  double val;
  if (lo && iy < c0) {
    val = lo[int64_t(iy - (c0 - g)) * nx1 + ix];
    b0[v] = val;
  } else if (up && iy > c1) {
    val = up[int64_t(iy - c1) * nx1 + ix];
    b0[v] = val;
  } else if (lo && iy == c0) {
    val = b0[v] + lo[int64_t(g) * nx1 + ix];
    b0[v] = val;
  } else if (up && iy == c1) {
    val = b0[v] + up[ix];
    b0[v] = val;
  } else {
    val = b0[v];
  }
  b1[v] = ((ix + iy) & 1) ? -val : val;
}

// The same for the nine coefficient arrays of the level-0 operator (once per solve): array e of lo / up starts at
// e (g + 1) nx1
__global__ void __launch_bounds__(kMgThreads)
    k_ghost_unpack_S(double* __restrict__ S, int64_t nv, const double* __restrict__ lo, const double* __restrict__ up, int nx, int c0,
                     int c1, int g, int lo_row, int hi_row) {
  const int nx1 = nx + 1;
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (tid >= int64_t(hi_row - lo_row + 1) * nx1) return;
  const int e = blockIdx.y;
  const int64_t v = int64_t(lo_row) * nx1 + tid;
  const int ix = int(v % nx1), iy = int(v / nx1);
  double* Se = S + int64_t(e) * nv;
  const int64_t chunk = int64_t(g + 1) * nx1;
  if (lo && iy < c0) Se[v] = lo[e * chunk + int64_t(iy - (c0 - g)) * nx1 + ix];
  else if (up && iy > c1) Se[v] = up[e * chunk + int64_t(iy - c1) * nx1 + ix];
  else if (lo && iy == c0) Se[v] += lo[e * chunk + int64_t(g) * nx1 + ix];
  else if (up && iy == c1) Se[v] += up[e * chunk + ix];
}

// ---- DG level on lattice-structured simplex grids: P = injection of the conforming P1 space (one hierarchy: the P1
// volume term is integrated exactly, there is no hourglass family) --------------------------------------------------------
// A_c = P^T A P per local vertex through the vertex -> DoF incidence of the Oswald pass; rows of cells owned elsewhere
// are added by the all-reduce
__global__ void __launch_bounds__(kMgThreads)
    k_vertex_galerkin_p1(MeshView m, const double* __restrict__ vals, const int64_t* __restrict__ vptr,
                         const int32_t* __restrict__ vdof, const int32_t* __restrict__ lvert_gid,
                         const int32_t* __restrict__ cell_gv, int32_t n_verts_loc, int nx, int ny, double* __restrict__ S) {
  const int lv = blockIdx.x * blockDim.x + threadIdx.x;
  if (lv >= n_verts_loc) return;
  const int nx1 = nx + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  const int v = __ldg(lvert_gid + lv);
  const int ix = v % nx1, iy = v / nx1;
  double acc[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) acc[e] = 0.0;
  bool any = false;
  for (int64_t q = __ldg(vptr + lv); q < __ldg(vptr + lv + 1); ++q) {
    const int dof = __ldg(vdof + q);
    const int c = dof / 3, i = dof - 3 * c, k = c - m.own0;
    if (k < 0 || k >= m.n_own) continue;
    any = true;
    int nb[3];
    nb[0] = __ldg(m.neigh + size_t(3) * k);
    nb[1] = __ldg(m.neigh + size_t(3) * k + 1);
    nb[2] = __ldg(m.neigh + size_t(3) * k + 2);
    const int nblk = block_count<3>(nb);
    const double* row = vals + __ldg(m.blk_start + k) * 9 + int64_t(i) * nblk * 3;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int cell = t == 0 ? c : nb[t - 1];
      if (cell < 0) continue;
      const int slot = block_slot<3>(c, nb, cell);
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int w = __ldg(cell_gv + size_t(3) * cell + j);
        const int dx = w % nx1 - ix, dy = w / nx1 - iy;
        if (dx < -1 || dx > 1 || dy < -1 || dy > 1) continue;  // cancels analytically (jumps of continuous functions)
        acc[(dy + 1) * 3 + dx + 1] += __ldg(row + slot * 3 + j);
      }
    }
  }
  if (!any) return;  // no owned cell at this vertex: its row comes from the owners
#pragma unroll
  for (int e = 0; e < 9; ++e) S[e * nv + v] = acc[e];
}

// b0 = P^T r: per local vertex the sum of the owned DG residual entries sitting on it
__global__ void __launch_bounds__(kMgThreads)
    k_dg_restrict_p1(const int* done, const double* __restrict__ r, const int64_t* __restrict__ vptr,
                     const int32_t* __restrict__ vdof, const int32_t* __restrict__ lvert_gid, int32_t n_verts_loc, int own0,
                     int n_own, double* __restrict__ b0) {
  if (done && *done) return;
  const int lv = blockIdx.x * blockDim.x + threadIdx.x;
  if (lv >= n_verts_loc) return;
  double s = 0.0;
  for (int64_t q = __ldg(vptr + lv); q < __ldg(vptr + lv + 1); ++q) {
    const int dof = __ldg(vdof + q);
    const int k = dof / 3 - own0;
    if (k < 0 || k >= n_own) continue;
    s += __ldg(r + size_t(dof) - size_t(3) * own0);
  }
  b0[__ldg(lvert_gid + lv)] = s;
}

// z += P x, r.z recomputed; optionally p = z (first direction).  One thread per owned triangle.
__global__ void __launch_bounds__(kMgThreads)
    k_dg_prolong_dot_p1(const int* done, int32_t n_cells, const int32_t* __restrict__ cell_gv /* of the owned cells */,
                        const double* __restrict__ x0, const double* __restrict__ r, double* __restrict__ z,
                        double* __restrict__ p_init, double* partial, CgScalars* sc) {
  if (done && *done) return;
  double v[1] = {0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; c < n_cells; c += stride) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double o = z[3 * c + i] + __ldg(x0 + __ldg(cell_gv + 3 * c + i));
      z[3 * c + i] = o;
      if (p_init) p_init[3 * c + i] = o;
      v[0] = fma(r[3 * c + i], o, v[0]);
    }
  }
  grid_sum<1>(v, partial, &sc->ticket_a, [sc](const double(&w)[1]) { sc->red[1] = w[0]; });
}

// ---- DG level for polOrder 2 on lattice-structured simplex grids ("cg.mg2.simplex"): P = interpolation of the conforming
// P1 space into P2-DG, one hierarchy (the P2 volume rule is exact: no hourglass family).  P2 nodes in the DoF order of
// Elem<SIMPLEX, 2>: (0,0), (1/2,0), (1,0), (0,1/2), (1/2,1/2), (0,1) - corner i of the cell is node p2_corner(i), the edge
// midpoints next to it are p2_mid1(i) and p2_mid2(i), each with weight 1/2 for either of its two corners.
__device__ __forceinline__ int p2_corner(int i) { return i == 0 ? 0 : i == 1 ? 2 : 5; }
__device__ __forceinline__ int p2_mid1(int i) { return i == 2 ? 3 : 1; }
__device__ __forceinline__ int p2_mid2(int i) { return i == 0 ? 3 : 4; }

// A_c = P^T A P per local vertex v: for every owned (cell, corner) at v the three rows of the nodes v interpolates into
// (its corner node with weight 1, the two adjacent edge midpoints with weight 1/2); each 6-wide block of such a row is
// folded onto the three vertices of the block's cell.  Entries at lattice distance 2 cancel analytically (jumps of
// continuous functions) and are dropped.  Writes only the rows of vertices with an owned triangle: the rows of cells owned
// elsewhere are added by the all-reduce.
__global__ void __launch_bounds__(kMgThreads)
    k_vertex_galerkin_p2(MeshView m, const double* __restrict__ vals, const int64_t* __restrict__ vptr,
                         const int32_t* __restrict__ vdof, const int32_t* __restrict__ lvert_gid,
                         const int32_t* __restrict__ cell_gv, int32_t n_verts_loc, int nx, int ny, double* __restrict__ S) {
  const int lv = blockIdx.x * blockDim.x + threadIdx.x;
  if (lv >= n_verts_loc) return;
  const int nx1 = nx + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  const int v = __ldg(lvert_gid + lv);
  const int ix = v % nx1, iy = v / nx1;
  double acc[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) acc[e] = 0.0;
  bool any = false;
  for (int64_t q = __ldg(vptr + lv); q < __ldg(vptr + lv + 1); ++q) {
    const int dof = __ldg(vdof + q);
    const int c = dof / 3, i = dof - 3 * c, k = c - m.own0;
    if (k < 0 || k >= m.n_own) continue;
    any = true;
    int nb[3];
    nb[0] = __ldg(m.neigh + size_t(3) * k);
    nb[1] = __ldg(m.neigh + size_t(3) * k + 1);
    nb[2] = __ldg(m.neigh + size_t(3) * k + 2);
    const int nblk = block_count<3>(nb);
    const double* blk = vals + __ldg(m.blk_start + k) * 36;
    const int rows[3] = {p2_corner(i), p2_mid1(i), p2_mid2(i)};
    const double wr[3] = {1.0, 0.5, 0.5};
#pragma unroll 1
    for (int t = 0; t < 4; ++t) {
      const int cell = t == 0 ? c : nb[t - 1];
      if (cell < 0) continue;
      const int slot = block_slot<3>(c, nb, cell);
      double f[3] = {0.0, 0.0, 0.0};  // the weighted rows folded onto vertex j of `cell`
#pragma unroll
      for (int rr = 0; rr < 3; ++rr) {
        const double* row = blk + int64_t(rows[rr]) * nblk * 6 + slot * 6;
        double a[6];
#pragma unroll
        for (int n = 0; n < 6; ++n) a[n] = __ldg(row + n);
        f[0] = fma(wr[rr], a[0] + 0.5 * (a[1] + a[3]), f[0]);
        f[1] = fma(wr[rr], a[2] + 0.5 * (a[1] + a[4]), f[1]);
        f[2] = fma(wr[rr], a[5] + 0.5 * (a[3] + a[4]), f[2]);
      }
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int w = __ldg(cell_gv + size_t(3) * cell + j);
        const int dx = w % nx1 - ix, dy = w / nx1 - iy;
        if (dx < -1 || dx > 1 || dy < -1 || dy > 1) continue;  // cancels analytically
        acc[(dy + 1) * 3 + dx + 1] += f[j];
      }
    }
  }
  if (!any) return;  // no owned cell at this vertex: its row comes from the owners
#pragma unroll
  for (int e = 0; e < 9; ++e) S[e * nv + v] = acc[e];
}

// b0 = P^T r: per local vertex, over the owned (cell, corner) pairs at it, r[corner node] + (r[mid 1] + r[mid 2]) / 2
__global__ void __launch_bounds__(kMgThreads)
    k_dg_restrict_p2(const int* done, const double* __restrict__ r, const int64_t* __restrict__ vptr,
                     const int32_t* __restrict__ vdof, const int32_t* __restrict__ lvert_gid, int32_t n_verts_loc, int own0,
                     int n_own, double* __restrict__ b0) {
  if (done && *done) return;
  const int lv = blockIdx.x * blockDim.x + threadIdx.x;
  if (lv >= n_verts_loc) return;
  double s = 0.0;
  for (int64_t q = __ldg(vptr + lv); q < __ldg(vptr + lv + 1); ++q) {
    const int dof = __ldg(vdof + q);
    const int c = dof / 3, i = dof - 3 * c, k = c - own0;
    if (k < 0 || k >= n_own) continue;
    const double* rc = r + size_t(6) * k;
    s += __ldg(rc + p2_corner(i)) + 0.5 * (__ldg(rc + p2_mid1(i)) + __ldg(rc + p2_mid2(i)));
  }
  b0[__ldg(lvert_gid + lv)] = s;
}

// z += P x, r.z recomputed; optionally p = z (first direction).  One thread per owned triangle, grid-stride.
__global__ void __launch_bounds__(kMgThreads)
    k_dg_prolong_dot_p2(const int* done, int32_t n_cells, const int32_t* __restrict__ cell_gv /* of the owned cells */,
                        const double* __restrict__ x0, const double* __restrict__ r, double* __restrict__ z,
                        double* __restrict__ p_init, double* partial, CgScalars* sc) {
  if (done && *done) return;
  double v[1] = {0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; c < n_cells; c += stride) {
    const double x[3] = {__ldg(x0 + __ldg(cell_gv + 3 * c)), __ldg(x0 + __ldg(cell_gv + 3 * c + 1)),
                         __ldg(x0 + __ldg(cell_gv + 3 * c + 2))};
    const double px[6] = {x[0], 0.5 * (x[0] + x[1]), x[1], 0.5 * (x[0] + x[2]), 0.5 * (x[1] + x[2]), x[2]};
#pragma unroll
    for (int n = 0; n < 6; ++n) {
      const double o = z[6 * c + n] + px[n];
      z[6 * c + n] = o;
      if (p_init) p_init[6 * c + n] = o;
      v[0] = fma(r[6 * c + n], o, v[0]);
    }
  }
  grid_sum<1>(v, partial, &sc->ticket_a, [sc](const double(&w)[1]) { sc->red[1] = w[0]; });
}

// lattice rows touched by the owned triangles: min / max of (vertex id / nx1) over their vertices
__global__ void k_vertex_row_range(const int32_t* __restrict__ gv_owned, int64_t n_entries, int nx1, int* __restrict__ minmax) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= n_entries) return;
  const int row = __ldg(gv_owned + t) / nx1;
  atomicMin(minmax, row);
  atomicMax(minmax + 1, row);
}

__global__ void k_cell_row_range(const int32_t* __restrict__ cell_v0_owned, int32_t n_own, int nx, int* __restrict__ minmax) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_own) return;
  const int cy = __ldg(cell_v0_owned + k) / (nx + 1);
  atomicMin(minmax, cy);
  atomicMax(minmax + 1, cy);
}

// z += P (x0 + C x1), r.z recomputed; optionally p = z (first direction).  One thread per cell, 256-bit accesses.
__global__ void __launch_bounds__(kMgThreads)
    k_dg_prolong_dot(const int* done, int32_t n_cells, const int32_t* __restrict__ cell_v0 /* of the owned cells */, int nx,
                     const double* __restrict__ x0, const double* __restrict__ x1, const double* __restrict__ r,
                     double* __restrict__ z, double* __restrict__ p_init, double* partial, CgScalars* sc) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  double v[1] = {0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; c < n_cells; c += stride) {
    const int v0 = __ldg(cell_v0 + c);
    const double sg = ((v0 % nx1 + v0 / nx1) & 1) ? -1.0 : 1.0;  // parity of vertex 0; vertices 1, 2 flip, 3 agrees
    const double4 zz = *reinterpret_cast<const double4*>(z + 4 * c);
    const double4 rr = *reinterpret_cast<const double4*>(r + 4 * c);
    double4 o;
    o.x = zz.x + __ldg(x0 + v0) + sg * __ldg(x1 + v0);
    o.y = zz.y + __ldg(x0 + v0 + 1) - sg * __ldg(x1 + v0 + 1);
    o.z = zz.z + __ldg(x0 + v0 + nx1) - sg * __ldg(x1 + v0 + nx1);
    o.w = zz.w + __ldg(x0 + v0 + nx1 + 1) + sg * __ldg(x1 + v0 + nx1 + 1);
    *reinterpret_cast<double4*>(z + 4 * c) = o;
    if (p_init) *reinterpret_cast<double4*>(p_init + 4 * c) = o;
    v[0] = fma(rr.x, o.x, fma(rr.y, o.y, fma(rr.z, o.z, fma(rr.w, o.w, v[0]))));
  }
  grid_sum<1>(v, partial, &sc->ticket_a, [sc](const double(&w)[1]) { sc->red[1] = w[0]; });
}

// ---- DG level for polOrder 2 on cubes ("cg.mg2"): two auxiliary vertex spaces with hierarchies of their own ----------
// P: bilinear interpolation of the conforming Q1 vertex space at the 9 nodes (node a + 3 b of a cell gets
//    q2_w(i, a) q2_w(j, b) of its vertex i + 2 j);
// H: the hourglass family - cell c gets s[v0(c)] q2_g(a) q2_g(b) at node a + 3 b, v0(c) its lower-left vertex.  Under the
//    2 x 2 Gauss rule of the Q2 volume term (x^2 - 1/3)(y^2 - 1/3) has a zero gradient at every quadrature point and is
//    continuous across faces: with a smooth amplitude it is an energy-free family no Q1 space represents (DESIGN.md 6).
// Hierarchy 0 holds A_P = P^T A P, hierarchy 1 A_H = H^T A H; both are 9-point vertex stencils.
__device__ __forceinline__ double q2_w(int i, int a) { return i == 0 ? 1.0 - 0.5 * a : 0.5 * a; }
__device__ __forceinline__ double q2_g(int a) { return a == 1 ? -1.0 / 3.0 : 2.0 / 3.0; }

// Both level-0 stencils per vertex v, gathered from the 9 x 9 blocks of the <= 4 owned cells around v (rows of cells owned
// elsewhere are added by the all-reduce).  A_P: the rows of the nodes v interpolates into, weighted towards the vertices of
// the block's cell (entries at index distance 2 cancel analytically, as for Q1).  A_H: only the cell whose lower-left
// vertex is v has hourglass rows at v; they couple to the face neighbours, whose lower-left vertices are lattice
// neighbours of v.  S: hierarchy 0 in S[e nv + v], hierarchy 1 in S[(9 + e) nv + v].
__global__ void __launch_bounds__(kMgThreads)
    k_vertex_galerkin_q2(MeshView m, const double* __restrict__ vals, const int32_t* __restrict__ cell_v0,
                         const int32_t* __restrict__ lex_cell, int nx, int ny, double* __restrict__ S) {
  const int64_t nv = int64_t(nx + 1) * (ny + 1);
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const int nx1 = nx + 1;
  const int ix = int(v % nx1), iy = int(v / nx1);
  double ap[9], ah[9];
#pragma unroll
  for (int e = 0; e < 9; ++e) ap[e] = ah[e] = 0.0;
#pragma unroll
  for (int b = 0; b < 2; ++b)
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int cx = ix - 1 + a, cy = iy - 1 + b;
      if (cx < 0 || cy < 0 || cx >= nx || cy >= ny) continue;
      const int c = __ldg(lex_cell + cx + nx * cy);
      const int k = c - m.own0;
      if (c < 0 || k < 0 || k >= m.n_own) continue;
      const int vx = 1 - a, vy = 1 - b;   // v is vertex vx + 2 vy of cell c
      const bool hg = a == 1 && b == 1;   // v is the lower-left vertex of c
      int nb[4];
      load_neigh4(m.neigh, k, nb);
      const int nblk = block_count<4>(nb);
      const double* blk = vals + __ldg(m.blk_start + k) * 81;
#pragma unroll 1
      for (int t = 0; t < 5; ++t) {
        const int cell = t == 0 ? c : nb[t - 1];
        if (cell < 0) continue;
        const int slot = block_slot<4>(c, nb, cell);
        const int v0 = __ldg(cell_v0 + cell);
        const int jx = v0 % nx1 - ix, jy = v0 / nx1 - iy;
        double sp[4] = {0.0, 0.0, 0.0, 0.0}, sh = 0.0;
#pragma unroll
        for (int n = 0; n < 9; ++n) {
          const double wp = q2_w(vx, n % 3) * q2_w(vy, n / 3);
          const double wh = hg ? q2_g(n % 3) * q2_g(n / 3) : 0.0;
          if (wp == 0.0 && wh == 0.0) continue;
          const double* row = blk + int64_t(n) * nblk * 9 + slot * 9;
          double rp[4] = {0.0, 0.0, 0.0, 0.0}, rh = 0.0;
#pragma unroll
          for (int q = 0; q < 9; ++q) {
            const double a_nq = __ldg(row + q);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const double w = q2_w(j & 1, q % 3) * q2_w(j >> 1, q / 3);
              if (w != 0.0) rp[j] = fma(w, a_nq, rp[j]);
            }
            rh = fma(q2_g(q % 3) * q2_g(q / 3), a_nq, rh);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) sp[j] = fma(wp, rp[j], sp[j]);
          sh = fma(wh, rh, sh);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int dx = jx + (j & 1), dy = jy + (j >> 1);
          if (dx < -1 || dx > 1 || dy < -1 || dy > 1) continue;
          ap[(dy + 1) * 3 + dx + 1] += sp[j];
        }
        if (hg) ah[(jy + 1) * 3 + jx + 1] += sh;
      }
    }
#pragma unroll
  for (int e = 0; e < 9; ++e) {
    S[e * nv + v] = ap[e];
    S[(9 + e) * nv + v] = ah[e];
  }
}

// No cell has its lower-left vertex in the top vertex row or the right vertex column: those rows of A_H are empty.  They
// get the mean diagonal of the other rows, which keeps the Jacobi sweeps and the coarsest Cholesky defined (the rows stay
// decoupled on level 0; H ignores their values).  One CTA, fixed summation order.
__global__ void __launch_bounds__(1024) k_hourglass_fill(double* __restrict__ diag, int nx, int ny) {
  __shared__ double smem[32];
  const int nx1 = nx + 1;
  const int64_t nv = int64_t(nx1) * (ny + 1);
  double s[1] = {0.0};
  for (int64_t v = threadIdx.x; v < nv; v += blockDim.x)
    if (v % nx1 < nx && v / nx1 < ny) s[0] += diag[v];
  block_sum<1>(s, smem);
  __shared__ double mean;
  if (threadIdx.x == 0) mean = s[0] / (double(nx) * ny);
  __syncthreads();
  for (int64_t v = threadIdx.x; v < nv; v += blockDim.x)
    if (v % nx1 == nx || v / nx1 == ny) diag[v] = mean;
}

// b_P = P^T r and b_H = H^T r: per vertex the weighted residual entries of the owned cells around it
__global__ void __launch_bounds__(kMgThreads)
    k_dg_restrict_q2(const int* done, const double* __restrict__ r, const int32_t* __restrict__ lex_cell, int own0, int n_own,
                     int nx, int ny, double* __restrict__ bp, double* __restrict__ bh) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  const int64_t v = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= int64_t(nx1) * (ny + 1)) return;
  const int ix = int(v % nx1), iy = int(v / nx1);
  double sp = 0.0, sh = 0.0;
#pragma unroll
  for (int b = 0; b < 2; ++b)
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int cx = ix - 1 + a, cy = iy - 1 + b;
      if (cx < 0 || cy < 0 || cx >= nx || cy >= ny) continue;
      const int k = __ldg(lex_cell + cx + nx * cy) - own0;
      if (k < 0 || k >= n_own) continue;
      const double* rc = r + size_t(9) * k;
      const int vx = 1 - a, vy = 1 - b;
#pragma unroll
      for (int n = 0; n < 9; ++n) {
        const double wp = q2_w(vx, n % 3) * q2_w(vy, n / 3);
        const bool hg = a == 1 && b == 1;
        if (wp == 0.0 && !hg) continue;
        const double rn = __ldg(rc + n);
        if (wp != 0.0) sp = fma(wp, rn, sp);
        if (hg) sh = fma(q2_g(n % 3) * q2_g(n / 3), rn, sh);
      }
    }
  bp[v] = sp;
  bh[v] = sh;
}

// z += P xp + H xh, r.z recomputed; optionally p = z (first direction).  One thread per owned cell.
__global__ void __launch_bounds__(kMgThreads)
    k_dg_prolong_dot_q2(const int* done, int32_t n_cells, const int32_t* __restrict__ cell_v0 /* of the owned cells */, int nx,
                        const double* __restrict__ xp, const double* __restrict__ xh, const double* __restrict__ r,
                        double* __restrict__ z, double* __restrict__ p_init, double* partial, CgScalars* sc) {
  if (done && *done) return;
  const int nx1 = nx + 1;
  double v[1] = {0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; c < n_cells; c += stride) {
    const int v0 = __ldg(cell_v0 + c);
    const double x[4] = {__ldg(xp + v0), __ldg(xp + v0 + 1), __ldg(xp + v0 + nx1), __ldg(xp + v0 + nx1 + 1)};
    const double h = __ldg(xh + v0);
#pragma unroll
    for (int n = 0; n < 9; ++n) {
      double o = z[9 * c + n];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double w = q2_w(j & 1, n % 3) * q2_w(j >> 1, n / 3);
        if (w != 0.0) o = fma(w, x[j], o);
      }
      o = fma(q2_g(n % 3) * q2_g(n / 3), h, o);
      z[9 * c + n] = o;
      if (p_init) p_init[9 * c + n] = o;
      v[0] = fma(r[9 * c + n], o, v[0]);
    }
  }
  grid_sum<1>(v, partial, &sc->ticket_a, [sc](const double(&w)[1]) { sc->red[1] = w[0]; });
}

}  // namespace

// ---- host side ------------------------------------------------------------------------------------------------
// One level of both hierarchies: the arrays of the twisted hierarchy follow those of the plain one (9 nv / nv entries
// behind).  Level 0 has one operator for both (C A_c C is A_c with the edge-neighbour entries negated).
struct MgLevel {
  int nx = 0, ny = 0;
  int64_t nv = 0;
  DevBuf<double> S, dinv, b, x, r, y;
  double* result = nullptr;  // where the level's correction ends up: y after post-smoothing, x on the coarsest level
};

constexpr int kMaxDist = 4;  // at most this many finest vertex levels are swept in row strips (ghost zones of 2, 8, 18, 38 rows)

// Multi GPU, cells in full-width bands of rows stacked in rank order: the vectors of the n_dist finest vertex levels are
// computed in row strips with ghost zones instead of exchanges.  Every array keeps its full size, so a vertex has the
// same index on every rank.  A rank receives the g rows of the level-0 right-hand side next to its strip once per
// application (one grouped send / recv with the ranks below and above) and then computes, redundantly, every value of
// the distributed levels its own rows depend on: the sweeps of level l run on the row ranges below, which shrink by one
// row per stencil application towards the rows this rank owns.  The values in the ghost zones are the same numbers the
// neighbour computes (same operations on the same data), so the result equals the replicated V-cycle.  The first
// replicated level gets its right-hand side by one all-reduce (every rank restricts into its own rows of a zeroed
// array); the operators are replicated (one all-reduce of the level-0 stencil per solve).
struct MgDist {
  bool on = false;
  int n_dist = 0;              // distributed levels 0 .. n_dist-1
  int lower = -1, upper = -1;  // ranks owning the strips below / above (-1: none)
  int c0 = 0, c1 = 0;          // owned cell rows [c0, c1) of level 0
  bool last = false;           // the top strip
  int ghost = 0;               // level-0 rows of b received from each neighbour
  // inclusive vertex-row ranges per distributed level: pre-smoothing (x, r), right-hand side b, post-smoothing (y),
  // prolongation (x += P x_H)
  int pre_lo[kMaxDist], pre_hi[kMaxDist], b_lo[kMaxDist], b_hi[kMaxDist], up_lo[kMaxDist], up_hi[kMaxDist],
      pro_lo[kMaxDist], pro_hi[kMaxDist];
  int own_lo = 0, own_hi = 0;  // own rows of the first replicated level (restricted into the all-reduced array)
  DevBuf<double> tmp_lo, tmp_up;
};

struct MgState {
  std::vector<std::unique_ptr<MgLevel>> levels;
  DevBuf<double> coarse_inv, coarse_work;  // [n_hier][n * n]: inverse of the coarsest operators, scratch of its computation
  DevBuf<int> coarse_flag;
  bool strips_known = false;
  int nx = 0, ny = 0;
  int n_hier = 2;  // Q1 on cubes: plain + checkerboard-twisted hierarchy; P1 on lattice-structured simplex grids: one
  // Q2 on cubes ("cg.mg2"): hierarchy 0 for A_P, hierarchy 1 for A_H, each with a level-0 operator of its own (the
  // twisted Q1 hierarchy instead reads its level-0 operator from the plain one's arrays)
  // P2 on lattice-structured simplex grids ("cg.mg2.simplex"): one hierarchy, as for P1
  MgKind kind = MgKind::mg;
  bool q2() const { return kind == MgKind::mg2; }
  MgDist dist;
};

static const char* mg_type_name(MgKind k) {
  return k == MgKind::mg2 ? "cg.mg2" : k == MgKind::mg2_simplex ? "cg.mg2.simplex" : "cg.mg";
}

static inline dim3 grid2(int64_t cnt, int n_hier = 2) { return dim3(unsigned(blocks_for(cnt)), unsigned(n_hier)); }

static inline Rows row_range(const MgLevel& L, int lo, int hi) {
  return Rows{int64_t(lo) * (L.nx + 1), int64_t(hi - lo + 1) * (L.nx + 1)};
}

// The row ranges of MgDist for the strip [c0, c1) of an ny-row grid with n_dist distributed levels (host arithmetic,
// exported for the CPU tests as hdd_mg_strip_plan).  Top-down: which rows of the post-smoothed correction, of the
// prolongated iterate and hence of the coarser correction are needed; bottom-up: which rows of the residual feed the
// restriction, hence of the pre-smoothing sweep and of the right-hand side.
void mg_strip_plan(int ny, int c0, int c1, int n_dist, MgDist& d) {
  const bool last = c1 == ny;
  auto clip = [](int v, int n) { return std::max(0, std::min(v, n)); };
  int need_lo = c0, need_hi = c1;  // rows of the level-0 correction the DG prolongation of the own cells reads
  for (int l = 0; l < n_dist; ++l) {
    const int n = ny >> l;
    d.up_lo[l] = clip(need_lo, n);
    d.up_hi[l] = clip(need_hi, n);
    d.pro_lo[l] = clip(d.up_lo[l] - 1, n);
    d.pro_hi[l] = clip(d.up_hi[l] + 1, n);
    need_lo = d.pro_lo[l] >> 1;
    need_hi = (d.pro_hi[l] + 1) >> 1;
  }
  // own rows of the first replicated level
  const int sh = n_dist;
  d.own_lo = c0 >> sh;
  d.own_hi = last ? (ny >> sh) : (c1 >> sh) - 1;
  int res_lo = d.own_lo, res_hi = d.own_hi;  // rows of level l+1 whose right-hand side this rank computes
  for (int l = n_dist - 1; l >= 0; --l) {
    const int n = ny >> l;
    const int rr_lo = clip(2 * res_lo - 1, n), rr_hi = clip(2 * res_hi + 1, n);  // residual rows the restriction reads
    d.pre_lo[l] = std::min(d.pro_lo[l], rr_lo);
    d.pre_hi[l] = std::max(d.pro_hi[l], rr_hi);
    d.b_lo[l] = clip(d.pre_lo[l] - 1, n);
    d.b_hi[l] = clip(d.pre_hi[l] + 1, n);
    res_lo = d.b_lo[l];
    res_hi = d.b_hi[l];
  }
  d.ghost = std::max(c0 - d.b_lo[0], d.b_hi[0] - c1);
}

// xy_dev is addressed by global vertex id and holds the vertices [v_begin, v_end) only (the ones the local cells touch):
// every rank checks its own cells and vertices; hdd_mesh_attach_comm makes the verdict collective.
void mg_detect_structure(hdd_mesh* m, const double* xy_host, const double* xy_dev, int64_t v_begin, int64_t v_end,
                         const int32_t* cv_dev, int64_t n_verts) {
  m->sx = m->sy = 0;
  m->lx = m->ly = 0;
  int64_t nx1 = 1;
  while (nx1 < n_verts && xy_host[2 * nx1 + 1] == xy_host[1]) ++nx1;
  if (nx1 < 2 || n_verts % nx1 != 0) return;
  const int64_t nx = nx1 - 1, ny = n_verts / nx1 - 1;
  cudaStream_t s = m->stream;
  if (m->kind == HDD_SIMPLEX2D) {
    // lattice-structured triangulation (two triangles per lattice cell, e.g. the ALU ladder): vertex coordinates are a
    // tensor product, every triangle joins lattice neighbours
    if (ny < 1 || 2 * nx * ny != m->n_global) return;
    std::vector<double> xs, ys;
    xs.resize(size_t(nx1));
    ys.resize(size_t(ny) + 1);
    for (int64_t i = 0; i < nx1; ++i) xs[size_t(i)] = xy_host[2 * i];
    for (int64_t j = 0; j <= ny; ++j) ys[size_t(j)] = xy_host[2 * j * nx1 + 1];
    DevBuf<double> d_xs, d_ys;
    d_xs.upload(xs.data(), xs.size(), s);
    d_ys.upload(ys.data(), ys.size(), s);
    DevBuf<int32_t> flag;
    flag.alloc(1);
    flag.zero(s);
    k_struct_triangles<<<blocks_for(m->n_loc), kMgThreads, 0, s>>>(cv_dev, m->n_loc, int(nx1), n_verts, flag.p);
    k_struct_verts<<<blocks_for(v_end - v_begin), kMgThreads, 0, s>>>(xy_dev, v_begin, v_end - v_begin, int(nx), d_xs.p, d_ys.p, flag.p);
    count_launch(2);
    int32_t f = 0;
    HDD_CUDA(cudaMemcpyAsync(&f, flag.p, sizeof(f), cudaMemcpyDeviceToHost, s));
    HDD_CUDA(cudaStreamSynchronize(s));
    if (f == 0) {
      m->lx = int(nx);
      m->ly = int(ny);
    }
    return;
  }
  if (ny < 1 || nx * ny != m->n_global) return;
  // column / row coordinates from the first grid row and the first grid column of the caller's array
  std::vector<double> xs, ys;
  xs.resize(size_t(nx1));
  ys.resize(size_t(ny) + 1);
  for (int64_t i = 0; i < nx1; ++i) xs[size_t(i)] = xy_host[2 * i];
  for (int64_t j = 0; j <= ny; ++j) ys[size_t(j)] = xy_host[2 * j * nx1 + 1];
  DevBuf<double> d_xs, d_ys;
  d_xs.upload(xs.data(), xs.size(), s);
  d_ys.upload(ys.data(), ys.size(), s);
  m->cell_v0.alloc(size_t(m->n_loc));
  m->lex_cell.alloc(size_t(m->n_global));
  HDD_CUDA(cudaMemsetAsync(m->lex_cell.p, 0xFF, size_t(m->n_global) * sizeof(int32_t), s));  // -1: not on this rank
  DevBuf<int32_t> flag;
  flag.alloc(1);
  flag.zero(s);
  k_struct_cells<<<blocks_for(m->n_loc), kMgThreads, 0, s>>>(cv_dev, m->n_loc, int(nx), int(ny), m->cell_v0.p, m->lex_cell.p, flag.p);
  k_struct_verts<<<blocks_for(v_end - v_begin), kMgThreads, 0, s>>>(xy_dev, v_begin, v_end - v_begin, int(nx), d_xs.p, d_ys.p, flag.p);
  m->tgeo.alloc(4 * size_t(nx + ny));
  k_struct_geo<<<blocks_for(nx + ny), kMgThreads, 0, s>>>(d_xs.p, d_ys.p, int(nx), int(ny), m->tgeo.p);
  count_launch(3);
  int32_t f = 0;
  HDD_CUDA(cudaMemcpyAsync(&f, flag.p, sizeof(f), cudaMemcpyDeviceToHost, s));
  HDD_CUDA(cudaStreamSynchronize(s));
  if (f != 0) {
    m->cell_v0.release();
    m->lex_cell.release();
    m->tgeo.release();
    return;
  }
  m->sx = int(nx);
  m->sy = int(ny);
}

// recomputes the Galerkin operators below the finest level and the dense coarsest inverses; the level buffers are
// allocated once per mesh by mg_setup and persist across solves, so a captured CUDA graph of the iteration stays valid.
// The twisted hierarchy has no level-0 arrays of its own: its finest operator is C A_c C, read from the level-0 arrays
// with the sign of the edge-neighbour entries flipped.
static void build_hierarchies(hdd_swipdg* h, MgState& st) {
  hdd_mesh* m = h->mesh;
  cudaStream_t s = m->stream;
  const size_t nl = st.levels.size();
  const MgDist& d = st.dist;
  const int nd = d.on ? d.n_dist : 0;
  // Strip mode: the operator of a distributed level is needed (and valid) on the rows of its right-hand side, b_lo .. b_hi;
  // the first replicated level is computed on the own rows and summed over the ranks, the levels below it are replicated.
  for (size_t l = 0; l + 1 < nl; ++l) {
    MgLevel& f = *st.levels[l];
    MgLevel& c = *st.levels[l + 1];
    Rows rc{0, c.nv};
    const int lc = int(l) + 1;
    const int nh = st.n_hier;
    if (lc < nd) {
      rc = row_range(c, d.b_lo[lc], d.b_hi[lc]);
    } else if (lc == nd && nd > 0) {
      HDD_CUDA(cudaMemsetAsync(c.S.p, 0, size_t(nh) * 9 * c.nv * sizeof(double), s));
      rc = row_range(c, d.own_lo, d.own_hi);
    }
    const bool shared = l == 0 && !st.q2();  // level 0 of the twisted hierarchy is read from the plain one's arrays
    k_rap<<<grid2(rc.cnt, nh), kMgThreads, 0, s>>>(f.S.p, shared ? 0 : 9 * f.nv, f.nx, f.ny, (shared && nh == 2) ? 1 : 0, rc, c.S.p,
                                                  9 * c.nv);
    count_launch();
    if (lc == nd && nd > 0) Nccl::get().all_reduce_sum(c.S.p, size_t(nh) * 9 * c.nv, m->comm, s);
  }
  for (size_t l = 0; l < nl; ++l) {
    MgLevel& L = *st.levels[l];
    const Rows r = int(l) < nd ? row_range(L, d.b_lo[l], d.b_hi[l]) : Rows{0, L.nv};
    k_mg_dinv<<<dim3(unsigned(blocks_for(r.cnt)), (l == 0 && !st.q2()) ? 1u : unsigned(st.n_hier)), kMgThreads, 0, s>>>(L.S.p, L.nv, r, L.dinv.p);
    count_launch();
  }
  // dense inverses of the coarsest operators (s.p.d.): Gauss-Jordan on the device, one CTA per hierarchy
  MgLevel& C = *st.levels.back();
  const char* type = mg_type_name(st.kind);
  if (C.nv > kMaxCoarse)
    HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET, type << ": the " << st.nx << " x " << st.ny << " grid cannot be coarsened by halving down to at most "
                                                           << kMaxCoarse << " vertices (stuck at " << C.nx << " x " << C.ny << ")");
  const int n = int(C.nv);
  const bool shared = nl == 1 && !st.q2();  // coarsest = finest level, whose operator the twisted hierarchy shares
  const size_t need = size_t(st.n_hier) * n * n;
  if (st.coarse_inv.n < need) st.coarse_inv.alloc(need);
  if (st.coarse_work.n < need) st.coarse_work.alloc(need);
  if (!st.coarse_flag.p) st.coarse_flag.alloc(1);
  st.coarse_flag.zero(s);
  // HDD_MG_COARSE_GJ=1: Gauss-Jordan instead of the banded Cholesky (A/B switch; also the fall-back for a band that does not
  // fit into shared memory - a long thin coarsest grid)
  static const bool gauss_jordan = [] { const char* e = std::getenv("HDD_MG_COARSE_GJ"); return e && e[0] == '1'; }();
  const size_t band_bytes = size_t(n) * size_t(C.nx + 3) * sizeof(double);
  if (!gauss_jordan && band_bytes <= 200 * 1024 && n <= 512) {
    HDD_CUDA(cudaFuncSetAttribute(k_dense_inverse_banded, cudaFuncAttributeMaxDynamicSharedMemorySize, int(band_bytes)));
    k_dense_inverse_banded<<<st.n_hier, 512, band_bytes, s>>>(C.S.p, shared ? 0 : int64_t(9) * n, C.nx, C.ny,
                                                              (shared && st.n_hier == 2) ? 1 : 0, st.coarse_work.p,
                                                              st.coarse_inv.p, st.coarse_flag.p);
  } else {
    k_dense_inverse<<<st.n_hier, 1024, 0, s>>>(C.S.p, shared ? 0 : int64_t(9) * n, C.nx, C.ny,
                                               (shared && st.n_hier == 2) ? 1 : 0, st.coarse_work.p, st.coarse_inv.p,
                                               st.coarse_flag.p);
  }
  count_launch();
  int bad = 0;
  HDD_CUDA(cudaMemcpyAsync(&bad, st.coarse_flag.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  HDD_CUDA(cudaStreamSynchronize(s));
  if (bad) HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET, type << ": the coarsest operator is not positive definite");
}

// levels with at most this many vertices prolongate and post-smooth in one kernel (launch bound there)
constexpr int64_t kFusedUpMaxVerts = 1500000;

// One V(1,1)-cycle of both hierarchies, right-hand sides in levels[0]->b (rows b_lo .. b_hi of this rank when the strip
// mode is on); the corrections end up in levels[0]->result.
static void vcycle(hdd_mesh* m, MgState& st, const int* done, cudaStream_t s) {
  const int nl = int(st.levels.size());
  const MgDist& d = st.dist;
  const int nd = d.on ? d.n_dist : 0;
  const int nh = st.n_hier;
  SolvePhases& pt = phase_timer();
  // ---- down: pre-smoothing + restriction ---------------------------------------------------------------------------
  for (int l = 0; l + 1 < nl; ++l) {
    MgLevel& L = *st.levels[size_t(l)];
    MgLevel& Cn = *st.levels[size_t(l) + 1];
    const Rows rp = l < nd ? row_range(L, d.pre_lo[l], d.pre_hi[l]) : Rows{0, L.nv};
    if (l == 0 && nh == 2 && !st.q2())
      k_mg_pre2<<<blocks_for(rp.cnt), kMgThreads, 0, s>>>(done, L.S.p, L.dinv.p, L.nx, L.ny, rp, L.b.p, L.x.p, L.r.p);
    else
      k_mg_pre<<<grid2(rp.cnt, nh), kMgThreads, 0, s>>>(done, L.S.p, L.dinv.p, L.nx, L.ny, rp, L.b.p, L.x.p, L.r.p);
    Rows rc{0, Cn.nv};
    if (l + 1 < nd) {
      rc = row_range(Cn, d.b_lo[l + 1], d.b_hi[l + 1]);
    } else if (l + 1 == nd && nd > 0) {
      // first replicated level: own rows into a zeroed array, summed over the ranks
      HDD_CUDA(cudaMemsetAsync(Cn.b.p, 0, size_t(nh) * Cn.nv * sizeof(double), s));
      rc = row_range(Cn, d.own_lo, d.own_hi);
    }
    k_mg_restrict<<<grid2(rc.cnt, nh), kMgThreads, 0, s>>>(done, L.r.p, L.nx, L.ny, rc, Cn.b.p);
    count_launch(2);
    pt.mark(l == 0 ? "mg down level 0" : l < nd ? "mg down distributed 1.." : "mg down replicated", s);
    if (l + 1 == nd && nd > 0) {
      Nccl::get().all_reduce_sum(Cn.b.p, size_t(nh) * Cn.nv, m->comm, s);
      pt.mark("mg all-reduce coarse rhs", s);
    }
  }
  // ---- coarsest: dense inverse ----------------------------------------------------------------------------------------
  MgLevel& C = *st.levels.back();
  k_mg_dense<<<dim3(unsigned(int(C.nv) + 3) / 4, unsigned(nh)), 128, 0, s>>>(done, st.coarse_inv.p, int(C.nv), C.b.p, C.x.p);
  count_launch();
  pt.mark("mg dense", s);
  C.result = C.x.p;
  // ---- up: prolongation + post-smoothing ----------------------------------------------------------------------------
  for (int l = nl - 2; l >= 0; --l) {
    MgLevel& L = *st.levels[size_t(l)];
    MgLevel& Cn = *st.levels[size_t(l) + 1];
    const Rows ru = l < nd ? row_range(L, d.up_lo[l], d.up_hi[l]) : Rows{0, L.nv};
    if (l > 0 && L.nv <= kFusedUpMaxVerts) {
      k_mg_up<<<grid2(ru.cnt, nh), kMgThreads, 0, s>>>(done, L.S.p, L.dinv.p, L.nx, L.ny, ru, L.b.p, L.x.p, Cn.result, L.y.p);
      count_launch();
    } else {
      const Rows rq = l < nd ? row_range(L, d.pro_lo[l], d.pro_hi[l]) : Rows{0, L.nv};
      k_mg_prolong_add<<<grid2(rq.cnt, nh), kMgThreads, 0, s>>>(done, Cn.result, L.nx, L.ny, rq, L.x.p);
      if (l == 0 && nh == 2 && !st.q2())
        k_mg_post2<<<blocks_for(ru.cnt), kMgThreads, 0, s>>>(done, L.S.p, L.dinv.p, L.nx, L.ny, ru, L.b.p, L.x.p, L.y.p);
      else
        k_mg_post<<<grid2(ru.cnt, nh), kMgThreads, 0, s>>>(done, L.S.p, L.dinv.p, L.nx, L.ny, ru, L.b.p, L.x.p, L.y.p);
      count_launch(2);
    }
    pt.mark(l == 0 ? "mg up level 0" : l < nd ? "mg up distributed 1.." : "mg up replicated", s);
    L.result = L.y.p;
  }
}

// Decides, identically on every rank, whether the ranks' cells are full-width bands of cell rows stacked in rank order
// whose boundaries and heights allow the strip mode, and with how many distributed levels (as many as kMaxDist).
// HDD_MG_DISTRIBUTED=0 keeps every vertex level replicated; HDD_MG_DIST_LEVELS=n caps the number of distributed levels.
static void detect_strips(hdd_swipdg* h, MgState& st) {
  hdd_mesh* m = h->mesh;
  MgDist& d = st.dist;
  d.on = false;
  d.n_dist = 0;
  static const bool wanted = [] { const char* e = std::getenv("HDD_MG_DISTRIBUTED"); return !(e && e[0] == '0'); }();
  static const int cap = [] { const char* e = std::getenv("HDD_MG_DIST_LEVELS"); return e ? std::atoi(e) : kMaxDist; }();
  if (m->world <= 1) return;
  cudaStream_t s = m->stream;
  DevBuf<int> mm;
  const int init[2] = {INT32_MAX, -1};
  mm.upload(init, 2, s);
  const bool cube = m->kind == HDD_CUBE2D;
  if (m->n_own > 0) {
    if (cube)
      k_cell_row_range<<<blocks_for(m->n_own), kMgThreads, 0, s>>>(m->cell_v0.p + m->own0, m->n_own, st.nx, mm.p);
    else
      k_vertex_row_range<<<blocks_for(int64_t(3) * m->n_own), kMgThreads, 0, s>>>(m->cell_gv.p + size_t(3) * m->own0,
                                                                                 int64_t(3) * m->n_own, st.nx + 1, mm.p);
  }
  count_launch();
  int got[2] = {0, 0};
  HDD_CUDA(cudaMemcpyAsync(got, mm.p, sizeof(got), cudaMemcpyDeviceToHost, s));
  HDD_CUDA(cudaStreamSynchronize(s));
  // cubes: cell rows [c0, c1); triangles: the lattice rows of their vertices are [c0, c1] - two triangles per lattice cell
  const int c0 = got[0], c1 = cube ? got[1] + 1 : got[1];
  const bool band = m->n_own > 0 && int64_t(m->n_own) == int64_t(cube ? 1 : 2) * st.nx * (c1 - c0);
  // every rank learns every rank's band: 3 doubles per rank through one all-reduce
  std::vector<double> all(size_t(3) * m->world, 0.0);
  all[size_t(3) * m->rank] = c0;
  all[size_t(3) * m->rank + 1] = c1;
  all[size_t(3) * m->rank + 2] = band ? 1.0 : 0.0;
  DevBuf<double> buf;
  buf.upload(all.data(), all.size(), s);
  Nccl::get().all_reduce_sum(buf.p, all.size(), m->comm, s);
  HDD_CUDA(cudaMemcpyAsync(all.data(), buf.p, all.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
  HDD_CUDA(cudaStreamSynchronize(s));
  if (!wanted) return;
  bool stacked = all[0] == 0.0 && all[size_t(3) * (m->world - 1) + 1] == double(st.ny);
  for (int r = 0; r < m->world; ++r) {
    stacked = stacked && all[size_t(3) * r + 2] == 1.0;
    if (r > 0) stacked = stacked && all[size_t(3) * r] == all[size_t(3) * (r - 1) + 1];
  }
  if (!stacked) return;
  // the largest number of distributed levels every band allows: boundaries on multiples of 2^n, enough rows for the
  // ghost zones to stay inside the adjacent strip, and at least one replicated level below
  int n_dist = 0;
  for (int n = std::min({cap, kMaxDist, int(st.levels.size()) - 1}); n >= 1 && n_dist == 0; --n) {
    bool ok = true;
    MgDist probe;
    mg_strip_plan(st.ny, 0, st.ny, n, probe);  // ghost width only depends on n away from the domain boundary
    for (int r = 0; r < m->world && ok; ++r) {
      const int a = int(all[size_t(3) * r]), b = int(all[size_t(3) * r + 1]);
      MgDist pr;
      mg_strip_plan(st.ny, a, b, n, pr);
      ok = a % (1 << n) == 0 && (b % (1 << n) == 0 || b == st.ny) && (b - a) >= 2 * pr.ghost + 2;
    }
    if (ok) n_dist = n;
  }
  if (n_dist == 0) return;
  d.on = true;
  d.n_dist = n_dist;
  d.c0 = c0;
  d.c1 = c1;
  d.lower = m->rank > 0 ? m->rank - 1 : -1;
  d.upper = m->rank + 1 < m->world ? m->rank + 1 : -1;
  d.last = d.upper < 0;
  mg_strip_plan(st.ny, c0, c1, n_dist, d);
  // the message size is the same on every rank: the ghost width of an interior strip
  MgDist interior;
  mg_strip_plan(st.ny, 1 << 20, (1 << 20) + (1 << 10), n_dist, interior);
  (void)interior;
  const size_t rows = size_t(d.ghost) + 1;
  if (d.tmp_lo.n < rows * (size_t(st.nx) + 1)) {
    d.tmp_lo.alloc(rows * (size_t(st.nx) + 1));
    d.tmp_up.alloc(rows * (size_t(st.nx) + 1));
  }
}

void mg_release(MgState* st) { delete st; }

// (re)builds the hierarchies for the frozen operator `vals`
void mg_setup(hdd_swipdg* h, const double* vals, MgKind kind) {
  hdd_mesh* m = h->mesh;
  const bool cube = m->kind == HDD_CUBE2D && m->sx > 0, lattice = m->kind == HDD_SIMPLEX2D && m->lx > 0;
  const bool q2 = kind == MgKind::mg2, p2s = kind == MgKind::mg2_simplex;
  const bool p2_lattice = lattice && h->polorder == 2;  // what "cg.mg2.simplex" is for
  if (q2 && h->polorder == 1)
    HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET, "solver type 'cg.mg2' is the multigrid preconditioner for polOrder 2; use 'cg.mg' for polOrder 1");
  if (q2 && !cube)
    HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET,
              "solver type 'cg.mg2' needs Q2 on a logically structured HDD_CUBE2D grid with the vertices numbered x-fastest "
              "(Stuff::Grid::Providers::Cube / hdd_grid_cube); use 'cg.blockdiagonal'"
                  << (p2_lattice ? " or 'cg.mg2.simplex'" : ""));
  if (p2s && m->kind != HDD_SIMPLEX2D)
    HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET,
              "solver type 'cg.mg2.simplex' needs a simplex grid; on HDD_CUBE2D grids use 'cg.mg' (polOrder 1) or 'cg.mg2' (polOrder 2)");
  if (p2s && h->polorder == 1)
    HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET,
              "solver type 'cg.mg2.simplex' is the multigrid preconditioner for polOrder 2 on triangles; use 'cg.mg' for polOrder 1");
  if (p2s && !lattice)
    HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET,
              "solver type 'cg.mg2.simplex' needs a simplex grid whose vertices form a lattice numbered x-fastest and whose "
              "triangles join lattice neighbours (the ALU ladder, hdd_grid_simplex); use 'cg.blockdiagonal'");
  if (kind == MgKind::mg && ((!cube && !lattice) || h->polorder != 1))
    HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET,
              "solver type 'cg.mg' needs polOrder 1 on a logically structured grid: HDD_CUBE2D with the vertices numbered x-fastest "
              "(Stuff::Grid::Providers::Cube / hdd_grid_cube) or a simplex grid whose vertices form such a lattice and whose "
              "triangles join lattice neighbours (the ALU ladder, hdd_grid_simplex); use 'cg.diagonal' or 'cg.blockdiagonal'"
                  << (p2_lattice ? " or 'cg.mg2.simplex'" : ""));
  cudaStream_t s = m->stream;
  if (!h->mg) h->mg = new MgState;
  MgState& st = *h->mg;
  st.nx = cube ? m->sx : m->lx;
  st.ny = cube ? m->sy : m->ly;
  st.n_hier = cube ? 2 : 1;
  st.kind = kind;
  const int64_t nv = int64_t(st.nx + 1) * (st.ny + 1);
  if (!st.levels.empty() && (st.levels[0]->nx != st.nx || st.levels[0]->ny != st.ny)) {
    st.levels.clear();
    st.strips_known = false;
  }
  if (st.levels.empty()) {  // level structure, allocation only
    int lx = st.nx, ly = st.ny;
    for (int l = 0;; ++l) {
      std::unique_ptr<MgLevel> L(new MgLevel);
      L->nx = lx;
      L->ny = ly;
      L->nv = int64_t(lx + 1) * (ly + 1);
      const size_t ops = (l == 0 && !q2) ? 1 : 2;  // the twisted hierarchy shares the level-0 operator of the plain one
      L->S.alloc(ops * 9 * size_t(L->nv));
      L->dinv.alloc(ops * size_t(L->nv));
      L->b.alloc(2 * size_t(L->nv));
      L->x.alloc(2 * size_t(L->nv));
      L->r.alloc(2 * size_t(L->nv));
      L->y.alloc(2 * size_t(L->nv));
      const bool last = L->nv <= kMaxCoarse || (lx & 1) || (ly & 1) || lx < 2 || ly < 2;
      st.levels.push_back(std::move(L));
      if (last) break;
      lx /= 2;
      ly /= 2;
    }
  }
  phase_timer().mark("setup mg: allocation", s);
  // the strip layout depends on the mesh and the communicator only: decided at the first solve of this discretization
  // (two stream synchronisations and a collective - 3 ms per solve at 2 and 8 ranks when repeated).  "cg.mg2" and
  // "cg.mg2.simplex" always run their vertex levels replicated.
  if (!st.strips_known && kind == MgKind::mg) {
    detect_strips(h, st);
    st.strips_known = true;
  }
  phase_timer().mark("setup mg: strip detection", s);
  MgLevel& f0 = *st.levels[0];
  const MgDist& d = st.dist;
  if (d.on) {
    // level-0 operator on the vertex rows of my cells (rows c0 and c1 are shared with the ranks below / above), then the
    // g rows next to the strip from the neighbours - instead of an all-reduce of the whole operator
    const int nx1 = st.nx + 1;
    const Rows mine{int64_t(d.c0) * nx1, int64_t(d.c1 - d.c0 + 1) * nx1};
    if (lattice)  // writes the rows of the vertices with an owned triangle: c0 .. c1
      k_vertex_galerkin_p1<<<blocks_for(m->n_verts_loc), kMgThreads, 0, s>>>(h->view(), vals, m->vptr.p, m->vdof.p, m->lvert_gid.p,
                                                                            m->cell_gv.p, m->n_verts_loc, st.nx, st.ny, f0.S.p);
    else
      k_vertex_galerkin<<<blocks_for(mine.cnt), kMgThreads, 0, s>>>(h->view(), vals, m->cell_v0.p, m->lex_cell.p, m->sx, m->sy, mine, f0.S.p);
    count_launch();
    const int g = d.ghost;
    const size_t chunk = size_t(g + 1) * nx1;
    DevBuf<double> lo, up;
    lo.alloc(9 * chunk);
    up.alloc(9 * chunk);
    Nccl& nc = Nccl::get();
    nc.group_start();
    for (int e = 0; e < 9; ++e) {
      double* Se = f0.S.p + int64_t(e) * nv;
      if (d.upper >= 0) {
        nc.send(Se + int64_t(d.c1 - g) * nx1, chunk, d.upper, m->comm, s);
        nc.recv(up.p + e * chunk, chunk, d.upper, m->comm, s);
      }
      if (d.lower >= 0) {
        nc.send(Se + int64_t(d.c0) * nx1, chunk, d.lower, m->comm, s);
        nc.recv(lo.p + e * chunk, chunk, d.lower, m->comm, s);
      }
    }
    nc.group_end();
    const int lo_row = d.b_lo[0], hi_row = d.b_hi[0];
    k_ghost_unpack_S<<<dim3(unsigned(blocks_for(int64_t(hi_row - lo_row + 1) * nx1)), 9u), kMgThreads, 0, s>>>(
        f0.S.p, nv, d.lower >= 0 ? lo.p : nullptr, d.upper >= 0 ? up.p : nullptr, st.nx, d.c0, d.c1, g, lo_row, hi_row);
    count_launch();
    HDD_CUDA(cudaStreamSynchronize(s));  // lo / up are freed at the end of this scope
  } else if (q2) {
    // every rank writes every vertex (zeros where it owns no cell): the all-reduce makes both operators global
    k_vertex_galerkin_q2<<<blocks_for(nv), kMgThreads, 0, s>>>(h->view(), vals, m->cell_v0.p, m->lex_cell.p, m->sx, m->sy, f0.S.p);
    count_launch();
    if (m->world > 1) Nccl::get().all_reduce_sum(f0.S.p, size_t(18) * nv, m->comm, s);
    k_hourglass_fill<<<1, 1024, 0, s>>>(f0.S.p + 13 * nv, st.nx, st.ny);  // diagonal of hierarchy 1: array 9 + 4
    count_launch();
  } else if (p2s) {
    if (m->world > 1) HDD_CUDA(cudaMemsetAsync(f0.S.p, 0, size_t(9) * nv * sizeof(double), s));
    k_vertex_galerkin_p2<<<blocks_for(m->n_verts_loc), kMgThreads, 0, s>>>(h->view(), vals, m->vptr.p, m->vdof.p, m->lvert_gid.p,
                                                                          m->cell_gv.p, m->n_verts_loc, st.nx, st.ny, f0.S.p);
    count_launch();
    if (m->world > 1) Nccl::get().all_reduce_sum(f0.S.p, size_t(9) * nv, m->comm, s);
  } else if (lattice) {
    if (m->world > 1) HDD_CUDA(cudaMemsetAsync(f0.S.p, 0, size_t(9) * nv * sizeof(double), s));
    k_vertex_galerkin_p1<<<blocks_for(m->n_verts_loc), kMgThreads, 0, s>>>(h->view(), vals, m->vptr.p, m->vdof.p, m->lvert_gid.p,
                                                                          m->cell_gv.p, m->n_verts_loc, st.nx, st.ny, f0.S.p);
    count_launch();
    if (m->world > 1) Nccl::get().all_reduce_sum(f0.S.p, size_t(9) * nv, m->comm, s);
  } else {
    k_vertex_galerkin<<<blocks_for(nv), kMgThreads, 0, s>>>(h->view(), vals, m->cell_v0.p, m->lex_cell.p, m->sx, m->sy, Rows{0, nv}, f0.S.p);
    count_launch();
    if (m->world > 1) Nccl::get().all_reduce_sum(f0.S.p, size_t(9) * nv, m->comm, s);
  }
  HDD_CUDA(cudaGetLastError());
  phase_timer().mark("setup mg: level-0 operator", s);
  build_hierarchies(h, st);
  phase_timer().mark("setup mg: coarse operators", s);
  HDD_CUDA(cudaGetLastError());
}

// z += P V(P^T r) + P C V_C(C P^T r) ("cg.mg2": z += P V_P(P^T r) + H V_H(H^T r); P1 on lattice simplices and
// "cg.mg2.simplex": z += P V(P^T r)), red[1] = r.z; p_init != nullptr also stores z as the first direction
void mg_apply(hdd_swipdg* h, const int* done, const double* r, double* z, double* p_init, double* partial, CgScalars* sc) {
  hdd_mesh* m = h->mesh;
  MgState& st = *h->mg;
  cudaStream_t s = m->stream;
  MgLevel& a = *st.levels[0];
  const bool multi = m->world > 1;
  const MgDist& d = st.dist;
  const int nx1 = st.nx + 1;
  double* b0 = a.b.p;
  double* b1 = a.b.p + a.nv;
  if (d.on) {
    // vertex rows c0 .. c1 of my cells; rows c0 and c1 are shared with the ranks below / above
    const Rows mine{int64_t(d.c0) * nx1, int64_t(d.c1 - d.c0 + 1) * nx1};
    if (st.n_hier == 1)  // triangles: every local vertex (rows c0 - 1 .. c1 + 1; the outer two receive zeros and are ghost rows)
      k_dg_restrict_p1<<<blocks_for(m->n_verts_loc), kMgThreads, 0, s>>>(done, r, m->vptr.p, m->vdof.p, m->lvert_gid.p, m->n_verts_loc,
                                                                        m->own0, m->n_own, b0);
    else
      k_dg_restrict<<<blocks_for(mine.cnt), kMgThreads, 0, s>>>(done, r, m->lex_cell.p, m->own0, m->n_own, st.nx, st.ny, mine, b0, nullptr);
    count_launch();
    phase_timer().mark("mg dg-restrict", s);
    const int g = d.ghost;
    const size_t cnt = size_t(g + 1) * nx1;
    Nccl& nc = Nccl::get();
    nc.group_start();
    if (d.upper >= 0) {
      nc.send(b0 + int64_t(d.c1 - g) * nx1, cnt, d.upper, m->comm, s);  // my rows [c1 - g, c1]
      nc.recv(d.tmp_up.p, cnt, d.upper, m->comm, s);                    // its rows [c1, c1 + g]
    }
    if (d.lower >= 0) {
      nc.send(b0 + int64_t(d.c0) * nx1, cnt, d.lower, m->comm, s);      // my rows [c0, c0 + g]
      nc.recv(d.tmp_lo.p, cnt, d.lower, m->comm, s);                    // its rows [c0 - g, c0]
    }
    nc.group_end();
    phase_timer().mark("mg ghost rows send/recv", s);
    const int lo_row = d.b_lo[0], hi_row = d.b_hi[0];
    k_ghost_unpack_twist<<<blocks_for(int64_t(hi_row - lo_row + 1) * nx1), kMgThreads, 0, s>>>(
        done, b0, b1, d.lower >= 0 ? d.tmp_lo.p : nullptr, d.upper >= 0 ? d.tmp_up.p : nullptr, st.nx, d.c0, d.c1, g, lo_row, hi_row);
    count_launch();
  } else if (st.kind == MgKind::mg2_simplex) {
    // P2 on a lattice-structured simplex grid: conforming P1 auxiliary space, one hierarchy, run replicated
    if (multi) HDD_CUDA(cudaMemsetAsync(b0, 0, size_t(a.nv) * sizeof(double), s));
    k_dg_restrict_p2<<<blocks_for(m->n_verts_loc), kMgThreads, 0, s>>>(done, r, m->vptr.p, m->vdof.p, m->lvert_gid.p, m->n_verts_loc,
                                                                      m->own0, m->n_own, b0);
    count_launch();
    if (multi) Nccl::get().all_reduce_sum(b0, size_t(a.nv), m->comm, s);
  } else if (st.q2()) {
    // Q2: b0 = P^T r, b1 = H^T r; every rank writes every vertex (zeros where it owns no cell), one all-reduce of both
    k_dg_restrict_q2<<<blocks_for(a.nv), kMgThreads, 0, s>>>(done, r, m->lex_cell.p, m->own0, m->n_own, st.nx, st.ny, b0, b1);
    count_launch();
    if (multi) Nccl::get().all_reduce_sum(b0, size_t(2) * a.nv, m->comm, s);
  } else if (st.n_hier == 1) {
    // lattice-structured simplex grid: conforming P1 auxiliary space, one hierarchy
    if (multi) HDD_CUDA(cudaMemsetAsync(b0, 0, size_t(a.nv) * sizeof(double), s));
    k_dg_restrict_p1<<<blocks_for(m->n_verts_loc), kMgThreads, 0, s>>>(done, r, m->vptr.p, m->vdof.p, m->lvert_gid.p, m->n_verts_loc,
                                                                      m->own0, m->n_own, b0);
    count_launch();
    if (multi) Nccl::get().all_reduce_sum(b0, size_t(a.nv), m->comm, s);
  } else {
    k_dg_restrict<<<blocks_for(a.nv), kMgThreads, 0, s>>>(done, r, m->lex_cell.p, m->own0, m->n_own, st.nx, st.ny, Rows{0, a.nv}, b0,
                                                           multi ? nullptr : b1);
    count_launch();
    if (multi) {
      Nccl::get().all_reduce_sum(b0, size_t(a.nv), m->comm, s);
      k_twist_vector<<<blocks_for(a.nv), kMgThreads, 0, s>>>(done, b0, st.nx, Rows{0, a.nv}, b1);
      count_launch();
    }
  }
  phase_timer().mark(d.on ? "mg ghost unpack" : "mg dg-restrict", s);
  if (st.levels.size() == 1) {
    // the fine vertex grid is already small enough for the dense solve
    k_mg_dense<<<dim3(unsigned(int(a.nv) + 3) / 4, unsigned(st.n_hier)), 128, 0, s>>>(done, st.coarse_inv.p, int(a.nv), a.b.p, a.x.p);
    count_launch();
    a.result = a.x.p;
  } else {
    vcycle(m, st, done, s);
  }
  const int grid = int(std::min<int64_t>((m->n_own + kMgThreads - 1) / kMgThreads, kMaxBlocks));
  if (st.q2())
    k_dg_prolong_dot_q2<<<grid, kMgThreads, 0, s>>>(done, m->n_own, m->cell_v0.p + m->own0, st.nx, a.result, a.result + a.nv, r, z,
                                                    p_init, partial, sc);
  else if (st.kind == MgKind::mg2_simplex)
    k_dg_prolong_dot_p2<<<grid, kMgThreads, 0, s>>>(done, m->n_own, m->cell_gv.p + size_t(3) * m->own0, a.result, r, z, p_init, partial, sc);
  else if (st.n_hier == 1)
    k_dg_prolong_dot_p1<<<grid, kMgThreads, 0, s>>>(done, m->n_own, m->cell_gv.p + size_t(3) * m->own0, a.result, r, z, p_init, partial, sc);
  else
    k_dg_prolong_dot<<<grid, kMgThreads, 0, s>>>(done, m->n_own, m->cell_v0.p + m->own0, st.nx, a.result, a.result + a.nv, r, z, p_init,
                                                 partial, sc);
  count_launch();
  phase_timer().mark("mg dg-prolong + r.z", s);
  HDD_CUDA(cudaGetLastError());
}

int mg_num_levels(const hdd_swipdg* h) { return h->mg ? int(h->mg->levels.size()) : 0; }

void mg_vertex_result(const hdd_swipdg* h, double* host) {
  const MgLevel& a = *h->mg->levels[0];
  HDD_CUDA(cudaMemcpyAsync(host, a.result, size_t(h->mg->n_hier) * a.nv * sizeof(double), cudaMemcpyDeviceToHost,
                           h->mesh->stream));
}

}  // namespace hdd

extern "C" int hdd_mg_level_operator(const hdd_swipdg* h, int level, int hier, int* nx, int* ny, double* S_host) {
  return hdd::guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    const hdd::MgState* st = h->mg;
    if (!st) HDD_THROW(HDD_ERR_USING_THIS_WRONG, "no multigrid hierarchy: solve with 'cg.mg', 'cg.mg2' or 'cg.mg2.simplex' first");
    if (level < 0 || level >= int(st->levels.size()))
      HDD_THROW(HDD_ERR_WRONG_INPUT, "level " << level << " of " << st->levels.size());
    if (hier < 0 || hier >= st->n_hier) HDD_THROW(HDD_ERR_WRONG_INPUT, "hierarchy " << hier << " of " << st->n_hier);
    if (level == 0 && hier == 1 && !st->q2())
      HDD_THROW(HDD_ERR_WRONG_INPUT, "level 0 of the twisted hierarchy is C A_c C, read from the plain one's arrays");
    const hdd::MgLevel& L = *st->levels[size_t(level)];
    if (nx) *nx = L.nx;
    if (ny) *ny = L.ny;
    if (S_host) {
      h->mesh->set_device();
      cudaStream_t s = h->mesh->stream;
      HDD_CUDA(cudaMemcpyAsync(S_host, L.S.p + size_t(hier) * 9 * L.nv, size_t(9) * L.nv * sizeof(double),
                               cudaMemcpyDeviceToHost, s));
      HDD_CUDA(cudaStreamSynchronize(s));
    }
  });
}

// host-only view of the strip plan for the CPU tests: out[8 * l + {0..7}] = pre_lo, pre_hi, b_lo, b_hi, up_lo, up_hi,
// pro_lo, pro_hi of level l; out[8 * n_dist + {0, 1, 2}] = own_lo, own_hi, ghost
extern "C" int hdd_mg_strip_plan(int ny, int c0, int c1, int n_dist, int* out) {
  if (!out || n_dist < 1 || n_dist > hdd::kMaxDist || c0 < 0 || c1 <= c0 || c1 > ny) return HDD_ERR_WRONG_INPUT;
  hdd::MgDist d;
  hdd::mg_strip_plan(ny, c0, c1, n_dist, d);
  for (int l = 0; l < n_dist; ++l) {
    const int v[8] = {d.pre_lo[l], d.pre_hi[l], d.b_lo[l], d.b_hi[l], d.up_lo[l], d.up_hi[l], d.pro_lo[l], d.pro_hi[l]};
    for (int k = 0; k < 8; ++k) out[8 * l + k] = v[k];
  }
  out[8 * n_dist] = d.own_lo;
  out[8 * n_dist + 1] = d.own_hi;
  out[8 * n_dist + 2] = d.ghost;
  return HDD_OK;
}
