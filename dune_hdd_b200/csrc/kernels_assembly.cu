// K1 (pattern), K2 (system matrix parts), K3 (rhs parts), K4 (freeze) for sm_100a.
//
// Assembly is owner-computes: one thread per owned cell produces the complete row block of that cell - its
// volume term, and for every face the en/en block (into the diagonal block) and the en/ne block (off-diagonal)
// seen with the cell's own outward normal.  The SWIPDG face terms are symmetric under swapping the roles of the
// two cells (omega^- <-> omega^+, n <-> -n; SURVEY 8a a5), so this reproduces what the reference's serial walk
// (system_assembler.walk(), discretizations/swipdg.hh:485) scatters into the rows of T from both sides, without
// atomics, colouring or a second pass, and bit-reproducibly.  A row block is one contiguous chunk of the CSR
// value array, written with 256-bit stores for Q1 (one full 32-byte sector per block row).
#include <cub/device/device_scan.cuh>

#include <cstring>

#include "kernels.hpp"

namespace hdd {

namespace {

constexpr int kThreads = 128;

inline int grid_for(int64_t n, int threads) { return int((n + threads - 1) / threads); }

template <int NF>
__device__ __forceinline__ void load_neigh(const int32_t* neigh, int k, int* nb) {
  if constexpr (NF == 4) {
    const int4 v = __ldg(reinterpret_cast<const int4*>(neigh) + k);
    nb[0] = v.x; nb[1] = v.y; nb[2] = v.z; nb[3] = v.w;
  } else {
#pragma unroll
    for (int f = 0; f < NF; ++f) nb[f] = __ldg(neigh + size_t(NF) * k + f);
  }
}

// xy is addressed by global vertex id and holds the vertices [v_begin, v_end) only
__global__ void k_build_geometry(int kind, int32_t n_loc, int32_t v_begin, int32_t v_end, const double* __restrict__ xy,
                                 const int32_t* __restrict__ cv, double* __restrict__ cgeo, int32_t* flag) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_loc) return;
  const double2* p = reinterpret_cast<const double2*>(xy);
  if (kind == HDD_SIMPLEX2D) {
    double2* out = reinterpret_cast<double2*>(cgeo + size_t(6) * c);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const int v = cv[size_t(3) * c + i];
      if (v < v_begin || v >= v_end) { atomicOr(flag, 4); return; }  // index validation happens here, not on the host
      out[i] = __ldg(p + v);
    }
  } else {
    const int4 v = __ldg(reinterpret_cast<const int4*>(cv) + c);
    if (v.x < v_begin || v.y < v_begin || v.z < v_begin || v.w < v_begin || v.x >= v_end || v.y >= v_end || v.z >= v_end ||
        v.w >= v_end) {
      atomicOr(flag, 4);
      return;
    }
    const double2 a = __ldg(p + v.x), b = __ldg(p + v.y), d = __ldg(p + v.z), e = __ldg(p + v.w);
    if (a.x != d.x || b.x != e.x || a.y != b.y || d.y != e.y) atomicOr(flag, 1);
    double2* out = reinterpret_cast<double2*>(cgeo + size_t(4) * c);
    out[0] = a;
    out[1] = e;
  }
}

// Structured cube grid with a px x py box partition, built on the device from closed forms (hdd_mesh_create_cube): one
// thread per local cell writes its geometry record, vertex 0, global id, the lexicographic -> local map and, for an
// owned cell, the global ids of its four face neighbours (translated to local ids by k_localize_neighbours afterwards).
// Coordinates are the expressions of the host generator (grids.cpp), so both paths give bit-identical geometry.
__device__ __forceinline__ int cube_cell_id(const CubeGridDesc& g, int i, int j) {
  if (i < 0 || j < 0 || i >= g.nx || j >= g.ny) return -1;
  int bx = 0, by = 0;
  while (bx + 1 < g.px && i >= g.X[bx + 1]) ++bx;
  while (by + 1 < g.py && j >= g.Y[by + 1]) ++by;
  const int w = g.X[bx + 1] - g.X[bx];
  return int(g.off[by * g.px + bx]) + (j - g.Y[by]) * w + (i - g.X[bx]);
}

__global__ void k_cube_fill(CubeGridDesc g, int32_t n_loc, int32_t own0, int32_t n_own, int32_t cell_begin,
                            const int32_t* __restrict__ halo /* sorted global ids: lower part, then upper part */,
                            double* __restrict__ cgeo, int32_t* __restrict__ cell_v0, int32_t* __restrict__ lex_cell,
                            int32_t* __restrict__ cgid, int32_t* __restrict__ neigh) {
  const int lc = blockIdx.x * blockDim.x + threadIdx.x;
  if (lc >= n_loc) return;
  const bool own = lc >= own0 && lc < own0 + n_own;
  const int gid = own ? cell_begin + (lc - own0) : halo[lc < own0 ? lc : lc - n_own];
  // subdomain of gid: binary search in the offsets, then the position inside the box
  int lo = 0, hi = g.px * g.py;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (g.off[mid] <= gid) lo = mid; else hi = mid;
  }
  const int bx = lo % g.px, by = lo / g.px;
  const int w = g.X[bx + 1] - g.X[bx];
  const int r = gid - int(g.off[lo]);
  const int i = g.X[bx] + r % w, j = g.Y[by] + r / w;
  double2* geo = reinterpret_cast<double2*>(cgeo + size_t(4) * lc);
  geo[0] = make_double2(g.x0 + (g.x1 - g.x0) * double(i) / double(g.nx), g.y0 + (g.y1 - g.y0) * double(j) / double(g.ny));
  geo[1] = make_double2(g.x0 + (g.x1 - g.x0) * double(i + 1) / double(g.nx), g.y0 + (g.y1 - g.y0) * double(j + 1) / double(g.ny));
  cell_v0[lc] = j * (g.nx + 1) + i;
  lex_cell[size_t(j) * g.nx + i] = lc;
  cgid[lc] = gid;
  if (own) {
    int4 nb;
    nb.x = cube_cell_id(g, i - 1, j);
    nb.y = cube_cell_id(g, i + 1, j);
    nb.z = cube_cell_id(g, i, j - 1);
    nb.w = cube_cell_id(g, i, j + 1);
    reinterpret_cast<int4*>(neigh)[lc - own0] = nb;
  }
}

// {x0, hx, 1/hx, -} per column followed by {y0, hy, 1/hy, -} per row, from the closed-form coordinates
__global__ void k_cube_tgeo(CubeGridDesc g, double* __restrict__ tgeo) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= g.nx + g.ny) return;
  double4* out = reinterpret_cast<double4*>(tgeo);
  if (t < g.nx) {
    const double a = g.x0 + (g.x1 - g.x0) * double(t) / double(g.nx), b = g.x0 + (g.x1 - g.x0) * double(t + 1) / double(g.nx);
    out[t] = make_double4(a, b - a, 1.0 / (b - a), 0.0);
  } else {
    const int r = t - g.nx;
    const double a = g.y0 + (g.y1 - g.y0) * double(r) / double(g.ny), b = g.y0 + (g.y1 - g.y0) * double(r + 1) / double(g.ny);
    out[t] = make_double4(a, b - a, 1.0 / (b - a), 0.0);
  }
}

// whole mesh on one GPU: neighbour ids are used as they are; range check and global ids = identity
__global__ void k_validate_neighbours(const int32_t* __restrict__ neigh, int64_t count, int32_t n_cells, int32_t* flag) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const int32_t g = neigh[t];
  if (g < -1 || g >= n_cells) atomicOr(flag, 8);
}

__global__ void k_iota(int32_t* __restrict__ out, int32_t n, int32_t first) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = first + t;
}

// subdomain structure of a whole mesh (grid::Multiscale view): offsets of the subdomain-major cell ranges, the
// neighbouring-subdomain relation as a byte matrix; flag |= 16 if the numbering is not subdomain-major
__global__ void k_subdomain_structure(const int32_t* __restrict__ sub, const int32_t* __restrict__ neigh, int nf,
                                      int32_t n_cells, int n_sub, int64_t* __restrict__ offsets, uint8_t* __restrict__ adj,
                                      int32_t* flag) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  const int s = sub[c];
  if (s < 0 || s >= n_sub) { atomicOr(flag, 16); return; }
  if (c + 1 < n_cells) {
    const int d = sub[c + 1] - s;
    if (d < 0 || d > 1) atomicOr(flag, 16);
    if (d == 1) offsets[s + 1] = c + 1;
  }
  for (int f = 0; f < nf; ++f) {
    const int g = neigh[size_t(nf) * c + f];
    if (g < 0 || g >= n_cells) continue;
    const int t = sub[g];
    if (t != s && t >= 0 && t < n_sub) adj[size_t(s) * n_sub + t] = 1;
  }
}

__global__ void k_localize_neighbours(int32_t* __restrict__ neigh, int64_t count, int32_t cb, int32_t ce,
                                      const int32_t* __restrict__ halo, int32_t n_lo, int32_t n_hi, int32_t* flag) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const int32_t g = neigh[t];
  if (g < 0) return;
  if (g >= cb && g < ce) { neigh[t] = n_lo + (g - cb); return; }
  // binary search in the sorted lower / upper halo list
  int lo = g < cb ? 0 : n_lo, hi = g < cb ? n_lo : n_lo + n_hi;
  const int base = lo, end = hi;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (halo[mid] < g) lo = mid + 1; else hi = mid;
  }
  if (lo >= end || halo[lo] != g) { atomicOr(flag, 2); return; }
  neigh[t] = g < cb ? lo : (ce - cb) + lo;  // upper halo follows the owned cells: n_lo + n_own + (lo - n_lo)
  (void)base;
}

__global__ void k_count_blocks(MeshView m, int64_t* __restrict__ nblk) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  const int nf = m.nf;
  int s = 1;
  for (int f = 0; f < nf; ++f) s += __ldg(m.neigh + size_t(nf) * k + f) >= 0 ? 1 : 0;
  nblk[k] = s;
}

template <int NF, int NL>
__global__ void k_fill_csr(MeshView m, int64_t* __restrict__ rowptr, int32_t* __restrict__ col) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= int64_t(m.n_own) * NL) return;
  const int k = int(t / NL), i = int(t % NL);
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  const int self = m.own0 + k;
  const int nblk = block_count<NF>(nb);
  const int64_t start = m.blk_start[k] * (NL * NL) + int64_t(i) * nblk * NL;
  rowptr[t] = start;
  if (t == int64_t(m.n_own) * NL - 1) rowptr[t + 1] = m.blk_start[m.n_own] * (NL * NL);
  auto write_block = [&](int slot, int g) {
    if constexpr (NL == 4) {  // one 16-byte store per block instead of four 4-byte ones
      *reinterpret_cast<int4*>(col + start + slot * 4) = make_int4(4 * g, 4 * g + 1, 4 * g + 2, 4 * g + 3);
    } else {
#pragma unroll
      for (int j = 0; j < NL; ++j) col[start + slot * NL + j] = NL * g + j;
    }
  };
  write_block(block_slot<NF>(self, nb, self), __ldg(m.cgid + self));
#pragma unroll
  for (int f = 0; f < NF; ++f)
    if (nb[f] >= 0) write_block(block_slot<NF>(self, nb, nb[f]), __ldg(m.cgid + nb[f]));
}

template <int NL>
__device__ __forceinline__ void store_block(double* __restrict__ row0, int row_stride, int slot, const double* B) {
#pragma unroll
  for (int i = 0; i < NL; ++i) {
    double* dst = row0 + size_t(i) * row_stride + slot * NL;
    if constexpr (NL == 4) {
      // one full 32-byte sector per block row (Blackwell 256-bit store, STG.E.ENL2.256)
      asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst), "d"(B[i * 4 + 0]), "d"(B[i * 4 + 1]),
                   "d"(B[i * 4 + 2]), "d"(B[i * 4 + 3])
                   : "memory");
    } else {
#pragma unroll
      for (int j = 0; j < NL; ++j) dst[j] = B[i * NL + j];
    }
  }
}

// Write-out of rows staged in shared memory: `total` doubles, element t of the CTA's contiguous range sits at stage[t] and
// goes to dst[t].  One elected thread hands the 16-byte aligned middle of the range to the bulk-copy engine
// (cp.async.bulk.global.shared::cta, SASS UBLKCP) instead of every thread looping over LDS + STG; the staging buffer is laid
// out so that shared and global addresses agree modulo 16 (the caller offsets its rows by `stage_pad(dst)` doubles).
// Must be called by every thread of the CTA after the rows have been written; returns when the shared memory may be reused.
__device__ __forceinline__ int stage_pad(const double* dst) { return int((reinterpret_cast<uintptr_t>(dst) >> 3) & 1); }

__device__ __forceinline__ void bulk_write_out(double* __restrict__ dst, const double* stage /* = stage0 + stage_pad(dst) */,
                                               int64_t total) {
  // make the generic-proxy writes to shared memory visible to the async proxy, then meet
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  const int head = stage_pad(dst);                       // elements in front of the first 16-byte boundary
  const int64_t body = total > head ? ((total - head) >> 1) << 1 : 0;
  if (threadIdx.x == 0 && body > 0) {
    const uint32_t src = uint32_t(__cvta_generic_to_shared(stage + head));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + head), "r"(src),
                 "r"(uint32_t(body * 8))
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  }
  if (threadIdx.x == 32 && head == 1 && total > 0) dst[0] = stage[0];
  if (threadIdx.x == 64 && head + body < total) dst[head + body] = stage[head + body];
}

// K2.  SURVEY 8a rows a4 (GDT::LocalEvaluation::Elliptic), a5 (SWIPDG::Inner), a6 (SWIPDG::BoundaryLHS).
// FK = kind of the diffusion-factor part (HDD_FN_*), resolved at compile time so that constant and cell-wise data
// cost no function evaluation per quadrature point.  An Expression is one global function: both sides of a face
// see the same value at the same point, so it is evaluated once per point.
__device__ __forceinline__ double expression_at(const DevFn& fn, double x, double y) {
  const double v[2] = {x, y};
  return eval_program(fn.prog, v);
}

template <int FK>
__device__ __forceinline__ double factor_at(const DevFn& fn, double a_cell, double x, double y) {
  if constexpr (FK == HDD_FN_EXPRESSION) return expression_at(fn, x, y);
  else return a_cell;
}

// P1 on triangles with an Expression factor.  Bounded for one resident CTA per SM it compiles without spills; bounded for 4
// it is squeezed to 128 registers with spilled values and measured slower (1.99 vs 1.92 ms on 16.8 M triangles).
__global__ void __launch_bounds__(kThreads, 1)
    k_assemble_lhs(MeshView m, const __grid_constant__ DevFn fn, ElemRule vol, LineRule fr, double s_in, double s_bnd,
                   double* __restrict__ vals) {
  using G = Geo<HDD_SIMPLEX2D>;
  constexpr int NL = G::NL, NF = G::NF;
  // P1 row blocks are 3 doubles wide: written straight from the registers every store instruction would touch 32
  // different sectors for 24 bytes each.  The row blocks of the CTA's cells are one contiguous range of the value array,
  // so they are staged in shared memory and written out as one bulk copy (see bulk_write_out).
  __shared__ __align__(16) double stage0[kThreads * (NF + 1) * NL * NL + 2];
  const int k_first = blockIdx.x * blockDim.x;
  const bool live = k_first + int(threadIdx.x) < m.n_own;
  const int k = live ? k_first + threadIdx.x : m.n_own - 1;  // idle threads of the last CTA recompute its last cell
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  const int nblk = block_count<NF>(nb);
  const int rs = nblk * NL;
  const int64_t base_blk = __ldg(m.blk_start + k_first);
  double* stage = stage0 + stage_pad(vals + base_blk * (NL * NL));
  double* row0 = stage + (m.blk_start[k] - base_blk) * (NL * NL);

  double D[NL * NL];
#pragma unroll
  for (int t = 0; t < NL * NL; ++t) D[t] = 0.0;

  // volume: sum_q w (a K grad phi_j) . grad phi_i, rule of order(a) + 2(p-1)  (no over-integration)
  for (int q = 0; q < vol.n; ++q) {
    double phi[NL], gx[NL], gy[NL], x, y;
    g.basis(vol.x[q], vol.y[q], phi, gx, gy);
    g.to_global(vol.x[q], vol.y[q], x, y);
    const double wa = vol.w[q] * g.detj * expression_at(fn, x, y);
#pragma unroll
    for (int j = 0; j < NL; ++j) {
      const double fx = wa * (K[0] * gx[j] + K[1] * gy[j]);
      const double fy = wa * (K[2] * gx[j] + K[3] * gy[j]);
#pragma unroll
      for (int i = 0; i < NL; ++i) D[i * NL + j] = fma(fx, gx[i], fma(fy, gy[i], D[i * NL + j]));
    }
  }

#pragma unroll 1
  for (int f = 0; f < NF; ++f) {
    const FaceGeo e = make_face(g, f);
    const int n = nb[f];
    // K n (own side) and delta^- = n . K n
    const double knx = K[0] * e.nx + K[2] * e.ny, kny = K[1] * e.nx + K[3] * e.ny;  // K^T n: (K grad phi).n = grad phi . K^T n
    const double dm = e.nx * (K[0] * e.nx + K[1] * e.ny) + e.ny * (K[2] * e.nx + K[3] * e.ny);
    if (n < 0) {
      if (m.btype && __ldg(m.btype + size_t(NF) * k + f) != 1) continue;
      // Dirichlet face: -(A grad phi_j . n) phi_i - phi_j (A grad phi_i . n) + pen phi_j phi_i
      const double pen0 = s_bnd * dm * e.ih;
      for (int q = 0; q < fr.n; ++q) {
        const double x = e.ax + fr.x[q] * (e.bx - e.ax), y = e.ay + fr.x[q] * (e.by - e.ay);
        double xi, eta, phi[NL], gx[NL], gy[NL], A[NL], B[NL];
        g.to_local(x, y, xi, eta);
        g.basis(xi, eta, phi, gx, gy);
        const double a = expression_at(fn, x, y);
        const double w = fr.w[q] * e.h;
        const double wpen = w * pen0 * a, wa = w * a;
#pragma unroll
        for (int i = 0; i < NL; ++i) {
          B[i] = wa * (gx[i] * knx + gy[i] * kny);  // w (A grad phi_i . n)
          A[i] = wpen * phi[i] - B[i];
        }
#pragma unroll
        for (int i = 0; i < NL; ++i)
#pragma unroll
          for (int j = 0; j < NL; ++j) D[i * NL + j] = fma(phi[i], A[j], fma(-B[i], phi[j], D[i * NL + j]));
      }
    } else {
      G gn;
      gn.load(m.cgeo, n);
      double Kn[4];
      load_tensor(m.tensor, n, Kn);
      const double knxp = Kn[0] * e.nx + Kn[2] * e.ny, knyp = Kn[1] * e.nx + Kn[3] * e.ny;
      const double dp = e.nx * (Kn[0] * e.nx + Kn[1] * e.ny) + e.ny * (Kn[2] * e.nx + Kn[3] * e.ny);
      const double isum = 1.0 / (dp + dm);
      const double gamma = dp * dm * isum;
      const double wm = dp * isum, wp = dm * isum;
      const double pen0 = s_in * gamma * 0.5 * e.ih;
      double E[NL * NL];
#pragma unroll
      for (int t = 0; t < NL * NL; ++t) E[t] = 0.0;
      for (int q = 0; q < fr.n; ++q) {
        const double x = e.ax + fr.x[q] * (e.bx - e.ax), y = e.ay + fr.x[q] * (e.by - e.ay);
        double xi, eta, phm[NL], php[NL], gx[NL], gy[NL], A[NL], B[NL], Cc[NL];
        const double a = expression_at(fn, x, y);  // the same value on both sides of the face
        const double w = fr.w[q] * e.h;
        const double wpen = w * pen0 * (a + a);
        const double wwm = w * wm * a, wwp = w * wp * a;
        g.to_local(x, y, xi, eta);
        g.basis(xi, eta, phm, gx, gy);
#pragma unroll
        for (int i = 0; i < NL; ++i) {
          B[i] = wwm * (gx[i] * knx + gy[i] * kny);  // w omega^- (A^- grad phi^-_i . n)
          A[i] = wpen * phm[i] - B[i];
        }
        gn.to_local(x, y, xi, eta);
        gn.basis(xi, eta, php, gx, gy);
#pragma unroll
        for (int j = 0; j < NL; ++j)
          Cc[j] = -wwp * (gx[j] * knxp + gy[j] * knyp) - wpen * php[j];  // -w omega^+ (A^+ grad phi^+_j . n) - w pen phi^+_j
#pragma unroll
        for (int i = 0; i < NL; ++i)
#pragma unroll
          for (int j = 0; j < NL; ++j) {
            D[i * NL + j] = fma(phm[i], A[j], fma(-B[i], phm[j], D[i * NL + j]));  // en/en
            E[i * NL + j] = fma(phm[i], Cc[j], fma(B[i], php[j], E[i * NL + j]));  // en/ne
          }
      }
      if (live) store_block<NL>(row0, rs, block_slot<NF>(c, nb, n), E);
    }
  }
  if (live) store_block<NL>(row0, rs, block_slot<NF>(c, nb, c), D);
  const int k_end = min(k_first + int(blockDim.x), m.n_own);
  bulk_write_out(vals + base_blk * (NL * NL), stage, (__ldg(m.blk_start + k_end) - base_blk) * (NL * NL));
}

// K2 for P1 on triangles with a diffusion factor that is constant per cell (Constant / per-cell data: ESV2007, SPE10,
// thermalblock).  Every integrand is then a polynomial of degree <= 2 along a face and constant in the cell, so the
// quadrature loops of k_assemble_lhs collapse into closed forms: with I_i = int_e phi_i = h/2 and M_ij = int_e phi_i phi_j
// = h/3, h/6 for the two nodes of the face (0 for the opposite one), b_i = omega a (grad phi_i . K^T n) constant,
//     en/en += pen M - I b^T - b I^T,      en/ne = -I b+^T - pen M+ + b I+^T
// (M+, I+ with the neighbour's basis: its node sitting on the same vertex).  Outward normal and face length come from the
// gradient of the opposite node's basis function: n = -grad phi_o / |grad phi_o|, h = 2 |T| |grad phi_o|.  Same integrals
// as the quadrature version to rounding; a third of the instructions and half the registers, so twice as many warps are
// resident to hide the neighbour gathers.
template <int FK, int P, int Q, int O>
__device__ __forceinline__ void p1_face(const MeshView& m, const DevFn& fn, const Geo<HDD_SIMPLEX2D>& g, const double* gx,
                                        const double* gy, const double* K, double area, double a_self, int k, int c, int n, int f,
                                        double s_in, double s_bnd, double* D, double* row0, int rs, const int* nb, bool live) {
  const double glen = sqrt(gx[O] * gx[O] + gy[O] * gy[O]);
  const double iglen = 1.0 / glen;
  const double nx = -gx[O] * iglen, ny = -gy[O] * iglen;
  const double h = 2.0 * area * glen;
  const double ktx = K[0] * nx + K[2] * ny, kty = K[1] * nx + K[3] * ny;  // K^T n
  const double dm = nx * (K[0] * nx + K[1] * ny) + ny * (K[2] * nx + K[3] * ny);
  const double h2 = 0.5 * h, h3 = h * (1.0 / 3.0), h6 = h * (1.0 / 6.0);
  if (n < 0) {
    if (m.btype && __ldg(m.btype + size_t(3) * k + f) != 1) return;
    const double pen = s_bnd * dm * a_self / h;
    double B[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) B[i] = a_self * (gx[i] * ktx + gy[i] * kty);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      D[P * 3 + j] -= h2 * B[j];
      D[Q * 3 + j] -= h2 * B[j];
      D[j * 3 + P] -= h2 * B[j];
      D[j * 3 + Q] -= h2 * B[j];
    }
    D[P * 3 + P] = fma(pen, h3, D[P * 3 + P]);
    D[Q * 3 + Q] = fma(pen, h3, D[Q * 3 + Q]);
    D[P * 3 + Q] = fma(pen, h6, D[P * 3 + Q]);
    D[Q * 3 + P] = fma(pen, h6, D[Q * 3 + P]);
    return;
  }
  Geo<HDD_SIMPLEX2D> gn;
  gn.load(m.cgeo, n);
  double Kn[4];
  load_tensor(m.tensor, n, Kn);
  double a_nb = a_self;
  if constexpr (FK == HDD_FN_CELLWISE) a_nb = __ldg(fn.cell + n);
  const double ktxp = Kn[0] * nx + Kn[2] * ny, ktyp = Kn[1] * nx + Kn[3] * ny;
  const double dp = nx * (Kn[0] * nx + Kn[1] * ny) + ny * (Kn[2] * nx + Kn[3] * ny);
  const double isum = 1.0 / (dp + dm);
  const double wm = dp * isum, wp = dm * isum;
  const double pen = s_in * dp * dm * isum * 0.5 * (a_self + a_nb) / h;
  double Bm[3], Bp[3];
  const double hx[3] = {-gn.i00 - gn.i10, gn.i00, gn.i10}, hy[3] = {-gn.i01 - gn.i11, gn.i01, gn.i11};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    Bm[i] = wm * a_self * (gx[i] * ktx + gy[i] * kty);
    Bp[i] = wp * a_nb * (hx[i] * ktxp + hy[i] * ktyp);
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    D[P * 3 + j] -= h2 * Bm[j];
    D[Q * 3 + j] -= h2 * Bm[j];
    D[j * 3 + P] -= h2 * Bm[j];
    D[j * 3 + Q] -= h2 * Bm[j];
  }
  D[P * 3 + P] = fma(pen, h3, D[P * 3 + P]);
  D[Q * 3 + Q] = fma(pen, h3, D[Q * 3 + Q]);
  D[P * 3 + Q] = fma(pen, h6, D[P * 3 + Q]);
  D[Q * 3 + P] = fma(pen, h6, D[Q * 3 + P]);
  // en/ne: rows P and Q see -h/2 b+_j - pen M+ + b_i I+_j, row O only b_O I+_j
  double E[9];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const bool onp = gn.vx[j] == g.vx[P] && gn.vy[j] == g.vy[P];
    const bool onq = gn.vx[j] == g.vx[Q] && gn.vy[j] == g.vy[Q];
    const double Ip = (onp || onq) ? h2 : 0.0;
    const double mp = onp ? h3 : onq ? h6 : 0.0, mq = onq ? h3 : onp ? h6 : 0.0;
    E[P * 3 + j] = -h2 * Bp[j] - pen * mp + Bm[P] * Ip;
    E[Q * 3 + j] = -h2 * Bp[j] - pen * mq + Bm[Q] * Ip;
    E[O * 3 + j] = Bm[O] * Ip;
  }
  if (live) store_block<3>(row0, rs, block_slot<3>(c, nb, n), E);
}

// 4 resident CTAs per SM: at most 128 registers and no spills; bounded for 5 it is squeezed to 96 registers and spills
template <int FK>
__global__ void __launch_bounds__(kThreads, 4)
    k_assemble_p1_closed(MeshView m, const __grid_constant__ DevFn fn, double s_in, double s_bnd, double* __restrict__ vals) {
  using G = Geo<HDD_SIMPLEX2D>;
  // row blocks are 3 doubles wide: staged in shared memory and written out as one bulk copy (see bulk_write_out)
  __shared__ __align__(16) double stage0[kThreads * 4 * 9 + 2];
  const int k_first = blockIdx.x * blockDim.x;
  const bool live = k_first + int(threadIdx.x) < m.n_own;
  const int k = live ? k_first + threadIdx.x : m.n_own - 1;
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  int nb[3];
  load_neigh<3>(m.neigh, k, nb);
  const int rs = block_count<3>(nb) * 3;
  const int64_t base_blk = __ldg(m.blk_start + k_first);
  double* dst = vals + base_blk * 9;
  double* stage = stage0 + stage_pad(dst);
  double* row0 = stage + (m.blk_start[k] - base_blk) * 9;
  double a_self = fn.value;
  if constexpr (FK == HDD_FN_CELLWISE) a_self = __ldg(fn.cell + c);
  const double gx[3] = {-g.i00 - g.i10, g.i00, g.i10}, gy[3] = {-g.i01 - g.i11, g.i01, g.i11};
  const double area = 0.5 * g.detj;
  double D[9];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const double fx = a_self * area * (K[0] * gx[j] + K[1] * gy[j]), fy = a_self * area * (K[2] * gx[j] + K[3] * gy[j]);
#pragma unroll
    for (int i = 0; i < 3; ++i) D[i * 3 + j] = fx * gx[i] + fy * gy[i];
  }
  p1_face<FK, 0, 1, 2>(m, fn, g, gx, gy, K, area, a_self, k, c, nb[0], 0, s_in, s_bnd, D, row0, rs, nb, live);
  p1_face<FK, 0, 2, 1>(m, fn, g, gx, gy, K, area, a_self, k, c, nb[1], 1, s_in, s_bnd, D, row0, rs, nb, live);
  p1_face<FK, 1, 2, 0>(m, fn, g, gx, gy, K, area, a_self, k, c, nb[2], 2, s_in, s_bnd, D, row0, rs, nb, live);
  if (live) store_block<3>(row0, rs, block_slot<3>(c, nb, c), D);
  const int k_end = min(k_first + int(blockDim.x), m.n_own);
  bulk_write_out(dst, stage, (__ldg(m.blk_start + k_end) - base_blk) * 9);
}

// K2 for Q1 on axis-parallel rectangles.  Same integrals as k_assemble_lhs, with two structural facts used at compile
// time per face F: only the two basis functions of the face's own nodes are non-zero on it (and only the two nodes of
// the neighbour's opposite face), and normals are +-e_x / +-e_y.  That halves the fp64 work (16 instead of 32 fused
// multiply-adds per block and quadrature point) and drops every sqrt / division from the face loop.
template <int F>
struct CubeFace {
  static constexpr bool vertical = F < 2;                 // faces 0,1: x = const; faces 2,3: y = const
  static constexpr double sgn = (F == 0 || F == 2) ? -1.0 : 1.0;
  static constexpr int a0 = F == 0 ? 0 : F == 1 ? 1 : F == 2 ? 0 : 2;  // own nodes on the face, in the direction of t
  static constexpr int a1 = F == 0 ? 2 : F == 1 ? 3 : F == 2 ? 1 : 3;
  static constexpr int b0 = F == 0 ? 1 : F == 1 ? 0 : F == 2 ? 2 : 0;  // neighbour's nodes on its opposite face
  static constexpr int b1 = F == 0 ? 3 : F == 1 ? 2 : F == 2 ? 3 : 1;
};

// reference gradients of Q1 at (xi, eta), scaled to physical: gx = d/dxi * ihx, gy = d/deta * ihy
__device__ __forceinline__ void q1_grads(double xi, double eta, double ihx, double ihy, double* gx, double* gy) {
  gx[0] = -(1.0 - eta) * ihx; gx[1] = (1.0 - eta) * ihx; gx[2] = -eta * ihx; gx[3] = eta * ihx;
  gy[0] = -(1.0 - xi) * ihy;  gy[1] = -xi * ihy;         gy[2] = (1.0 - xi) * ihy; gy[3] = xi * ihy;
}

template <int F, int FK>
__device__ __forceinline__ void cube_face(const MeshView& m, const DevFn& fn, const Geo<HDD_CUBE2D>& g, const double* K,
                                          int k, int c, int n, double nb_ihx, double nb_ihy, double a_self,
                                          const LineRule& fr, double s_in, double s_bnd, double* D, double* row0, int rs,
                                          const int* nb) {
  using CF = CubeFace<F>;
  constexpr int NL = 4;
  const double h = CF::vertical ? fabs(g.hy) : fabs(g.hx);
  const double ih = CF::vertical ? fabs(g.ihy) : fabs(g.ihx);
  const double knx = CF::sgn * (CF::vertical ? K[0] : K[2]);  // (K^T n)_x
  const double kny = CF::sgn * (CF::vertical ? K[1] : K[3]);
  const double dm = CF::vertical ? K[0] : K[3];              // n . K n
  const double xi_own = CF::vertical ? (F == 1 ? 1.0 : 0.0) : 0.0, eta_own = CF::vertical ? 0.0 : (F == 3 ? 1.0 : 0.0);
  if (n < 0) {
    if (m.btype && __ldg(m.btype + size_t(4) * k + F) != 1) return;
    const double pen0 = s_bnd * dm * ih;
    for (int q = 0; q < fr.n; ++q) {
      const double t = fr.x[q];
      const double xi = CF::vertical ? xi_own : t, eta = CF::vertical ? t : eta_own;
      double gx[NL], gy[NL], B[NL];
      q1_grads(xi, eta, g.ihx, g.ihy, gx, gy);
      double a = a_self;
      if constexpr (FK == HDD_FN_EXPRESSION) a = factor_at<FK>(fn, a_self, g.x0 + g.hx * xi, g.y0 + g.hy * eta);
      const double w = fr.w[q] * h, wa = w * a, wpen = w * pen0 * a;
      const double p0 = 1.0 - t, p1 = t;
#pragma unroll
      for (int i = 0; i < NL; ++i) B[i] = wa * (gx[i] * knx + gy[i] * kny);
      // D[i][j] += phi_i A_j - B_i phi_j with A_j = wpen phi_j - B_j; phi is non-zero at a0, a1 only
#pragma unroll
      for (int j = 0; j < NL; ++j) {
        const double Aj = (j == CF::a0 ? wpen * p0 : j == CF::a1 ? wpen * p1 : 0.0) - B[j];
        D[CF::a0 * NL + j] = fma(p0, Aj, D[CF::a0 * NL + j]);
        D[CF::a1 * NL + j] = fma(p1, Aj, D[CF::a1 * NL + j]);
      }
#pragma unroll
      for (int i = 0; i < NL; ++i) {
        D[i * NL + CF::a0] = fma(-B[i], p0, D[i * NL + CF::a0]);
        D[i * NL + CF::a1] = fma(-B[i], p1, D[i * NL + CF::a1]);
      }
    }
    return;
  }
  double Kn[4];
  load_tensor(m.tensor, n, Kn);
  const double knxp = CF::sgn * (CF::vertical ? Kn[0] : Kn[2]);
  const double knyp = CF::sgn * (CF::vertical ? Kn[1] : Kn[3]);
  const double dp = CF::vertical ? Kn[0] : Kn[3];
  const double isum = 1.0 / (dp + dm);
  const double gamma = dp * dm * isum, wm = dp * isum, wp = dm * isum;
  const double pen0 = s_in * gamma * 0.5 * ih;
  double a_nb = a_self;
  if constexpr (FK == HDD_FN_CELLWISE) a_nb = __ldg(fn.cell + n);
  // the neighbour sees the face from its opposite side
  const double xi_nb = CF::vertical ? (F == 0 ? 1.0 : 0.0) : 0.0, eta_nb = CF::vertical ? 0.0 : (F == 2 ? 1.0 : 0.0);
  double E[NL * NL];
#pragma unroll
  for (int t2 = 0; t2 < NL * NL; ++t2) E[t2] = 0.0;
  for (int q = 0; q < fr.n; ++q) {
    const double t = fr.x[q];
    const double xi = CF::vertical ? xi_own : t, eta = CF::vertical ? t : eta_own;
    double gx[NL], gy[NL], B[NL], Cc[NL];
    double am = a_self;
    if constexpr (FK == HDD_FN_EXPRESSION) am = factor_at<FK>(fn, a_self, g.x0 + g.hx * xi, g.y0 + g.hy * eta);
    const double ap = (FK == HDD_FN_EXPRESSION) ? am : a_nb;
    const double w = fr.w[q] * h;
    const double wpen = w * pen0 * (am + ap), wwm = w * wm * am, wwp = w * wp * ap;
    const double p0 = 1.0 - t, p1 = t;
    q1_grads(xi, eta, g.ihx, g.ihy, gx, gy);
#pragma unroll
    for (int i = 0; i < NL; ++i) B[i] = wwm * (gx[i] * knx + gy[i] * kny);
    q1_grads(CF::vertical ? xi_nb : t, CF::vertical ? t : eta_nb, nb_ihx, nb_ihy, gx, gy);
#pragma unroll
    for (int j = 0; j < NL; ++j)
      Cc[j] = -wwp * (gx[j] * knxp + gy[j] * knyp) - (j == CF::b0 ? wpen * p0 : j == CF::b1 ? wpen * p1 : 0.0);
#pragma unroll
    for (int j = 0; j < NL; ++j) {
      const double Aj = (j == CF::a0 ? wpen * p0 : j == CF::a1 ? wpen * p1 : 0.0) - B[j];
      D[CF::a0 * NL + j] = fma(p0, Aj, D[CF::a0 * NL + j]);      // en/en: phi^-_i A_j
      D[CF::a1 * NL + j] = fma(p1, Aj, D[CF::a1 * NL + j]);
      E[CF::a0 * NL + j] = fma(p0, Cc[j], E[CF::a0 * NL + j]);   // en/ne: phi^-_i C_j
      E[CF::a1 * NL + j] = fma(p1, Cc[j], E[CF::a1 * NL + j]);
    }
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      D[i * NL + CF::a0] = fma(-B[i], p0, D[i * NL + CF::a0]);   // en/en: -B_i phi^-_j
      D[i * NL + CF::a1] = fma(-B[i], p1, D[i * NL + CF::a1]);
      E[i * NL + CF::b0] = fma(B[i], p0, E[i * NL + CF::b0]);    // en/ne: +B_i phi^+_j
      E[i * NL + CF::b1] = fma(B[i], p1, E[i * NL + CF::b1]);
    }
  }
  store_block<NL>(row0, rs, block_slot<4>(c, nb, n), E);
}

// The row block of one Q1 cell from its already loaded records (neighbour ids, block offset, vertex 0).
// TENSOR: the mesh is a logically structured tensor grid (MeshView::tgeo): the cell sizes of the cell and of its four
// neighbours come from the one-dimensional column / row tables (a few KB, cache resident) instead of the per-cell
// geometry records - no dependent neigh -> cgeo[neighbour] round trip, 160 bytes less gather traffic per cell.
template <int FK, bool TENSOR>
__device__ __forceinline__ void assemble_cube_cell(const MeshView& m, const DevFn& fn, const ElemRule& vol, const LineRule& fr,
                                                   double s_in, double s_bnd, double* __restrict__ vals, int k, const int* nb,
                                                   int64_t blk, int v0) {
  using G = Geo<HDD_CUBE2D>;
  constexpr int NL = 4, NF = 4;
  const int c = m.own0 + k;
  G g;
  double nihx[NF], nihy[NF];
  if constexpr (TENSOR) {
    const int cx = v0 % (m.tnx + 1), cy = v0 / (m.tnx + 1);
    const double* tx = m.tgeo;                      // 4 doubles per column: x0, hx, 1/hx, -
    const double* ty = m.tgeo + 4 * size_t(m.tnx);  // 4 doubles per row:    y0, hy, 1/hy, -
    const double2 ox = __ldg(reinterpret_cast<const double2*>(tx + 4 * cx));
    const double2 oy = __ldg(reinterpret_cast<const double2*>(ty + 4 * cy));
    g.x0 = ox.x; g.hx = ox.y; g.x1 = ox.x + ox.y; g.ihx = __ldg(tx + 4 * cx + 2);
    g.y0 = oy.x; g.hy = oy.y; g.y1 = oy.x + oy.y; g.ihy = __ldg(ty + 4 * cy + 2);
    g.detj = fabs(g.hx * g.hy);
    // left / right neighbours share the row, bottom / top neighbours the column
    nihx[0] = __ldg(tx + 4 * max(cx - 1, 0) + 2);
    nihx[1] = __ldg(tx + 4 * min(cx + 1, m.tnx - 1) + 2);
    nihx[2] = nihx[3] = g.ihx;
    nihy[0] = nihy[1] = g.ihy;
    nihy[2] = __ldg(ty + 4 * max(cy - 1, 0) + 2);
    nihy[3] = __ldg(ty + 4 * min(cy + 1, m.tny - 1) + 2);
  } else {
    g.load(m.cgeo, c);
  }
  double K[4];
  load_tensor(m.tensor, c, K);
  const int nblk = block_count<NF>(nb);
  const int rs = nblk * NL;
  double* row0 = vals + blk * (NL * NL);
  double a_self = 0.0;
  if constexpr (FK == HDD_FN_CONSTANT) a_self = fn.value;
  if constexpr (FK == HDD_FN_CELLWISE) a_self = __ldg(fn.cell + c);
  if constexpr (!TENSOR) {
    // all four neighbour records are requested up front: one memory latency instead of four in the face loop
    double2 lo[NF], hi[NF];
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      const double2* p = reinterpret_cast<const double2*>(m.cgeo + size_t(4) * (nb[f] >= 0 ? nb[f] : c));
      lo[f] = __ldg(p);
      hi[f] = __ldg(p + 1);
    }
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      nihx[f] = 1.0 / (hi[f].x - lo[f].x);
      nihy[f] = 1.0 / (hi[f].y - lo[f].y);
    }
  }
  double D[NL * NL];
#pragma unroll
  for (int t = 0; t < NL * NL; ++t) D[t] = 0.0;
  for (int q = 0; q < vol.n; ++q) {
    double gx[NL], gy[NL];
    q1_grads(vol.x[q], vol.y[q], g.ihx, g.ihy, gx, gy);
    const double wa = vol.w[q] * g.detj *
                      factor_at<FK>(fn, a_self, g.x0 + g.hx * vol.x[q], g.y0 + g.hy * vol.y[q]);
#pragma unroll
    for (int j = 0; j < NL; ++j) {
      const double fx = wa * (K[0] * gx[j] + K[1] * gy[j]);
      const double fy = wa * (K[2] * gx[j] + K[3] * gy[j]);
#pragma unroll
      for (int i = 0; i < NL; ++i) D[i * NL + j] = fma(fx, gx[i], fma(fy, gy[i], D[i * NL + j]));
    }
  }
  cube_face<0, FK>(m, fn, g, K, k, c, nb[0], nihx[0], nihy[0], a_self, fr, s_in, s_bnd, D, row0, rs, nb);
  cube_face<1, FK>(m, fn, g, K, k, c, nb[1], nihx[1], nihy[1], a_self, fr, s_in, s_bnd, D, row0, rs, nb);
  cube_face<2, FK>(m, fn, g, K, k, c, nb[2], nihx[2], nihy[2], a_self, fr, s_in, s_bnd, D, row0, rs, nb);
  cube_face<3, FK>(m, fn, g, K, k, c, nb[3], nihx[3], nihy[3], a_self, fr, s_in, s_bnd, D, row0, rs, nb);
  store_block<NL>(row0, rs, block_slot<NF>(c, nb, c), D);
}

template <int FK, int MINB, bool TENSOR>
__global__ void __launch_bounds__(kThreads, MINB)
    k_assemble_lhs_cube(MeshView m, const __grid_constant__ DevFn fn, ElemRule vol, LineRule fr, double s_in, double s_bnd,
                        double* __restrict__ vals) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  int nb[4];
  load_neigh<4>(m.neigh, k, nb);
  const int v0 = TENSOR ? __ldg(m.cell_v0 + m.own0 + k) : 0;
  assemble_cube_cell<FK, TENSOR>(m, fn, vol, fr, s_in, s_bnd, vals, k, nb, m.blk_start[k], v0);
}

// select v[i] for a run-time i without dynamic register indexing
template <int N>
__device__ __forceinline__ double pick(const double* v, int i) {
  double r = v[0];
#pragma unroll
  for (int k = 1; k < N; ++k) r = (k == i) ? v[k] : r;
  return r;
}

// K2, generic in the polynomial order: one thread per matrix ROW (cell k, test function i).  Used for p = 2, where a
// whole n_loc x n_loc block pair per thread (162 doubles for Q2) would not fit the register file, and for the penalty
// product.  Same integrals and the same owner-computes argument as k_assemble_lhs; the n_loc threads of a cell repeat
// the basis evaluation (cheap next to the 8 B/nnz they have to write).
//   MODE 0: the SWIPDG bilinear form (volume + inner + Dirichlet faces)
//   MODE 1: only its penalty terms - Products::SwipdgPenaltyAssemblable (discretizations/swipdg.hh:444-479)
template <int KIND, int P, int FK, int MODE, int MINB = 2>
__global__ void __launch_bounds__(kThreads, MINB)
    k_assemble_rows(MeshView m, const __grid_constant__ DevFn fn, ElemRule vol, LineRule fr, double s_in, double s_bnd,
                    double* __restrict__ vals) {
  using G = Elem<KIND, P>;
  constexpr int NL = G::NL, NF = G::NF;
  // The rows of the CTA are one contiguous range of the value array.  Written straight from the registers every store
  // instruction would touch 32 sectors for 8 bytes each (four partial writes per sector: the L2 request rate, not the
  // fp64 pipe, bounded the first version); the rows are staged in shared memory and written out as one bulk copy instead.
  __shared__ __align__(16) double stage0[kThreads * (NF + 1) * NL + 2];
  const int64_t n_rows = int64_t(m.n_own) * NL;
  const int64_t t_first = int64_t(blockIdx.x) * blockDim.x;
  const bool live = t_first + threadIdx.x < n_rows;
  const int64_t t = live ? t_first + threadIdx.x : n_rows - 1;  // idle threads of the last CTA recompute its last row
  const int k = int(t / NL), i = int(t % NL);
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  const int nblk = block_count<NF>(nb);
  int64_t base;  // first value of the CTA's first row
  {
    const int kf = int(t_first / NL), jf = int(t_first % NL);
    int nbf[NF];
    load_neigh<NF>(m.neigh, kf, nbf);
    base = __ldg(m.blk_start + kf) * (NL * NL) + int64_t(jf) * block_count<NF>(nbf) * NL;
  }
  const int64_t row_off = m.blk_start[k] * (NL * NL) + int64_t(i) * nblk * NL;
  double* stage = stage0 + stage_pad(vals + base);
  double* row = stage + (row_off - base);
  double a_self = 0.0;
  if constexpr (FK == HDD_FN_CONSTANT) a_self = fn.value;
  if constexpr (FK == HDD_FN_CELLWISE) a_self = __ldg(fn.cell + c);

  double D[NL];
#pragma unroll
  for (int j = 0; j < NL; ++j) D[j] = 0.0;

  if constexpr (MODE == 0) {
    for (int q = 0; q < vol.n; ++q) {
      double phi[NL], gx[NL], gy[NL], x, y;
      g.basis(vol.x[q], vol.y[q], phi, gx, gy);
      g.to_global(vol.x[q], vol.y[q], x, y);
      const double wa = vol.w[q] * g.detj * factor_at<FK>(fn, a_self, x, y);
      const double gxi = wa * pick<NL>(gx, i), gyi = wa * pick<NL>(gy, i);
#pragma unroll
      for (int j = 0; j < NL; ++j)
        D[j] = fma(K[0] * gx[j] + K[1] * gy[j], gxi, fma(K[2] * gx[j] + K[3] * gy[j], gyi, D[j]));
    }
  }

#pragma unroll 1
  for (int f = 0; f < NF; ++f) {
    const FaceGeo e = make_face(g, f);
    const int n = nb[f];
    const double knx = K[0] * e.nx + K[2] * e.ny, kny = K[1] * e.nx + K[3] * e.ny;
    const double dm = e.nx * (K[0] * e.nx + K[1] * e.ny) + e.ny * (K[2] * e.nx + K[3] * e.ny);
    if (n < 0) {
      if (m.btype && __ldg(m.btype + size_t(NF) * k + f) != 1) continue;
      const double pen0 = s_bnd * dm * e.ih;
      for (int q = 0; q < fr.n; ++q) {
        const double x = e.ax + fr.x[q] * (e.bx - e.ax), y = e.ay + fr.x[q] * (e.by - e.ay);
        double xi, eta, phi[NL], gx[NL], gy[NL];
        g.to_local(x, y, xi, eta);
        g.basis(xi, eta, phi, gx, gy);
        const double a = factor_at<FK>(fn, a_self, x, y);
        const double w = fr.w[q] * e.h;
        const double wpen = w * pen0 * a, wa = w * a;
        const double phii = pick<NL>(phi, i);
        if constexpr (MODE == 0) {
          const double Bi = wa * (pick<NL>(gx, i) * knx + pick<NL>(gy, i) * kny);
#pragma unroll
          for (int j = 0; j < NL; ++j) {
            const double Aj = wpen * phi[j] - wa * (gx[j] * knx + gy[j] * kny);
            D[j] = fma(phii, Aj, fma(-Bi, phi[j], D[j]));
          }
        } else {
#pragma unroll
          for (int j = 0; j < NL; ++j) D[j] = fma(phii * wpen, phi[j], D[j]);
        }
      }
    } else {
      G gn;
      gn.load(m.cgeo, n);
      double Kn[4];
      load_tensor(m.tensor, n, Kn);
      const double knxp = Kn[0] * e.nx + Kn[2] * e.ny, knyp = Kn[1] * e.nx + Kn[3] * e.ny;
      const double dp = e.nx * (Kn[0] * e.nx + Kn[1] * e.ny) + e.ny * (Kn[2] * e.nx + Kn[3] * e.ny);
      const double isum = 1.0 / (dp + dm);
      const double gamma = dp * dm * isum;
      const double wm = dp * isum, wp = dm * isum;
      const double pen0 = s_in * gamma * 0.5 * e.ih;
      double a_nb = a_self;
      if constexpr (FK == HDD_FN_CELLWISE) a_nb = __ldg(fn.cell + n);
      double E[NL];
#pragma unroll
      for (int j = 0; j < NL; ++j) E[j] = 0.0;
      for (int q = 0; q < fr.n; ++q) {
        const double x = e.ax + fr.x[q] * (e.bx - e.ax), y = e.ay + fr.x[q] * (e.by - e.ay);
        double xi, eta, ph[NL], gx[NL], gy[NL];
        const double am = factor_at<FK>(fn, a_self, x, y);
        const double ap = (FK == HDD_FN_EXPRESSION) ? am : a_nb;
        const double w = fr.w[q] * e.h;
        const double wpen = w * pen0 * (am + ap);
        const double wwm = w * wm * am, wwp = w * wp * ap;
        g.to_local(x, y, xi, eta);
        g.basis(xi, eta, ph, gx, gy);
        const double phii = pick<NL>(ph, i);
        double Bi = 0.0;
        if constexpr (MODE == 0) {
          Bi = wwm * (pick<NL>(gx, i) * knx + pick<NL>(gy, i) * kny);
#pragma unroll
          for (int j = 0; j < NL; ++j) {
            const double Aj = wpen * ph[j] - wwm * (gx[j] * knx + gy[j] * kny);
            D[j] = fma(phii, Aj, fma(-Bi, ph[j], D[j]));                       // en/en
          }
        } else {
#pragma unroll
          for (int j = 0; j < NL; ++j) D[j] = fma(phii * wpen, ph[j], D[j]);
        }
        gn.to_local(x, y, xi, eta);
        gn.basis(xi, eta, ph, gx, gy);
        if constexpr (MODE == 0) {
#pragma unroll
          for (int j = 0; j < NL; ++j) {
            const double Cj = -wwp * (gx[j] * knxp + gy[j] * knyp) - wpen * ph[j];
            E[j] = fma(phii, Cj, fma(Bi, ph[j], E[j]));                         // en/ne
          }
        } else {
#pragma unroll
          for (int j = 0; j < NL; ++j) E[j] = fma(-phii * wpen, ph[j], E[j]);
        }
      }
      if (live) {
        double* dst = row + block_slot<NF>(c, nb, n) * NL;
#pragma unroll
        for (int j = 0; j < NL; ++j) dst[j] = E[j];
      }
    }
  }
  if (live) {
    double* dst = row + block_slot<NF>(c, nb, c) * NL;
#pragma unroll
    for (int j = 0; j < NL; ++j) dst[j] = D[j];
  }
  // end of the CTA's last row
  const int64_t t_last = min(t_first + int64_t(blockDim.x), n_rows) - 1;
  const int kl = int(t_last / NL), il = int(t_last % NL);
  int nbl[NF];
  load_neigh<NF>(m.neigh, kl, nbl);
  const int nblkl = block_count<NF>(nbl);
  const int64_t total = __ldg(m.blk_start + kl) * (NL * NL) + int64_t(il + 1) * nblkl * NL - base;
  bulk_write_out(vals + base, stage, total);
}

// K2 for Q2 on axis-parallel rectangles (BASELINE config 5 at p = 2).  One thread per matrix row, 32 cells per CTA.
// What makes the generic row kernel fp64-bound is that the nine row threads of a cell each re-evaluate the nine basis
// functions and their fluxes at every face point.  Here (a) the basis is the tensor product l_a(xi) l_b(eta) of the
// quadratic Lagrange polynomials, so everything needed on a face follows from three values l(t_q) and three derivatives
// along the face plus the constants l(0), l(1), l'(0), l'(1) across it, and only the three functions of the face's own
// nodes are non-zero on it; (b) the two vectors that couple all nine columns,
//     A_j = w pen phi_j - w omega^- (A^- grad phi_j . n)        (en/en)
//     C_j = -w omega^+ (A^+ grad phi^+_j . n) - w pen phi^+_j     (en/ne)
// do not depend on the row: thread j of a cell computes A_j, C_j for the three face points once and the nine row threads
// read them from shared memory.  A row then costs 24 fused multiply-adds per face point instead of ~350 fp64 operations.
// The rows of a CTA's cells are one contiguous range of the value array: they are staged in shared memory and written out
// coalesced (written straight from the registers every store instruction touches 32 sectors for 8 bytes each, and the L2
// request rate - 1.7 G partial-sector writes for 13.6 GB at 2048^2 - bounds the kernel: measured 12.7 ms).
constexpr int kQ2Cells = 16;
constexpr int kQ2Threads = kQ2Cells * 9;
constexpr int kQ2MaxFacePts = 4;
constexpr int kQ2TabDoubles = 2 * kQ2Cells * kQ2MaxFacePts * 2 * 9;  // A_j, C_j of two faces in flight
constexpr int kQ2StageDoubles = kQ2Cells * 5 * 81;                    // every block of every cell of the CTA
constexpr int kQ2SmemBytes = (kQ2TabDoubles + kQ2StageDoubles + 2) * 8;

__host__ __device__ __forceinline__ void lagrange2(double t, double* l, double* d) {
  l[0] = (1.0 - t) * (1.0 - 2.0 * t); l[1] = 4.0 * t * (1.0 - t); l[2] = t * (2.0 * t - 1.0);
  d[0] = 4.0 * t - 3.0;               d[1] = 4.0 - 8.0 * t;       d[2] = 4.0 * t - 1.0;
}

template <int F>
__device__ __forceinline__ void q2_face(const MeshView& m, const DevFn& fn, const Geo<HDD_CUBE2D>& g, const double* K, int k,
                                        int c, int n, int i, const LineRule& fr, double s_in, double s_bnd,
                                        double* tab /* this cell's [q][2][9] */, double* D, double* row, const int* nb, bool live) {
  constexpr bool vertical = F < 2;                      // faces 0,1: x = const; faces 2,3: y = const
  constexpr double sgn = (F == 0 || F == 2) ? -1.0 : 1.0;
  constexpr int side = (F == 1 || F == 3) ? 2 : 0;      // index of the 1-d node on the face: own side, neighbour's 2 - side
  const int ai = i % 3, bi = i / 3;
  const int across = vertical ? ai : bi, along = vertical ? bi : ai;
  // l and l' across the face at the face coordinate (0 or 1): l = unit vector, l' = (-3, 4, -1) or (1, -4, 3)
  const double dl_own = side == 0 ? (across == 0 ? -3.0 : across == 1 ? 4.0 : -1.0) : (across == 0 ? 1.0 : across == 1 ? -4.0 : 3.0);
  const double dl_nb = side == 0 ? (across == 0 ? 1.0 : across == 1 ? -4.0 : 3.0) : (across == 0 ? -3.0 : across == 1 ? 4.0 : -1.0);
  const double l_own = across == side ? 1.0 : 0.0, l_nb = across == 2 - side ? 1.0 : 0.0;
  const double h = vertical ? fabs(g.hy) : fabs(g.hx);
  const double ih = vertical ? fabs(g.ihy) : fabs(g.ihx);
  const double i_across = vertical ? g.ihx : g.ihy, i_along = vertical ? g.ihy : g.ihx;
  // (K^T n) split into the across / along components of the face
  const double kn_ac = sgn * (vertical ? K[0] : K[3]), kn_al = sgn * (vertical ? K[1] : K[2]);
  const double dm = vertical ? K[0] : K[3];
  const bool inner = n >= 0;
  const bool dirichlet = !inner && !(m.btype && __ldg(m.btype + size_t(4) * k + F) != 1);
  double wm = 1.0, wp = 0.0, pen0 = s_bnd * dm * ih, kn_ac_p = 0.0, kn_al_p = 0.0, i_across_p = 0.0;
  if (inner) {
    double Kn[4];
    load_tensor(m.tensor, n, Kn);
    const double dp = vertical ? Kn[0] : Kn[3];
    const double isum = 1.0 / (dp + dm);
    wm = dp * isum;
    wp = dm * isum;
    pen0 = s_in * dp * dm * isum * 0.5 * ih;
    kn_ac_p = sgn * (vertical ? Kn[0] : Kn[3]);
    kn_al_p = sgn * (vertical ? Kn[1] : Kn[2]);
    Geo<HDD_CUBE2D> gn;
    gn.load(m.cgeo, n);
    i_across_p = vertical ? gn.ihx : gn.ihy;
  }
  // ---- phase 1: this thread's column j = i of A and C at every face point; its own B_i and phi_i stay in registers
  double Bi[kQ2MaxFacePts], phi_i[kQ2MaxFacePts];
  for (int q = 0; q < fr.n; ++q) {
    double lt[3], dt[3];
    lagrange2(fr.x[q], lt, dt);
    const double xi = vertical ? (side == 0 ? 0.0 : 1.0) : fr.x[q], eta = vertical ? fr.x[q] : (side == 0 ? 0.0 : 1.0);
    const double a = expression_at(fn, g.x0 + g.hx * xi, g.y0 + g.hy * eta);  // the same on both sides
    const double w = fr.w[q] * h;
    const double wpen = inner ? w * pen0 * (a + a) : w * pen0 * a;
    const double wwm = w * wm * a, wwp = w * wp * a;
    const double la = pick<3>(lt, along), da = pick<3>(dt, along);
    const double phi = l_own * la;
    // grad phi . K^T n = d/d(across) * kn_ac + d/d(along) * kn_al
    const double B = wwm * (dl_own * la * i_across * kn_ac + l_own * da * i_along * kn_al);
    double A = wpen * phi - B, C = 0.0;
    if (!inner && !dirichlet) A = 0.0;
    if (inner) {
      const double phip = l_nb * la;
      C = -wwp * (dl_nb * la * i_across_p * kn_ac_p + l_nb * da * i_along * kn_al_p) - wpen * phip;
    }
    tab[(q * 2 + 0) * 9 + i] = A;
    tab[(q * 2 + 1) * 9 + i] = C;
    Bi[q] = (inner || dirichlet) ? B : 0.0;
    phi_i[q] = (inner || dirichlet) ? phi : 0.0;
  }
  __syncthreads();
  // ---- phase 2: row i.  D[j] += phi_i A_j - B_i phi_j ; E[j] = phi_i C_j + B_i phi^+_j ; phi_j, phi^+_j are non-zero for the
  // three nodes on the face only (values l(t_q))
  double E[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) E[j] = 0.0;
  for (int q = 0; q < fr.n; ++q) {
    double lt[3], dt[3];
    lagrange2(fr.x[q], lt, dt);
    const double* A = tab + (q * 2 + 0) * 9;
    const double* C = tab + (q * 2 + 1) * 9;
    const double p = phi_i[q], B = Bi[q];
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      D[j] = fma(p, A[j], D[j]);
      E[j] = fma(p, C[j], E[j]);
    }
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const int j_own = vertical ? side + 3 * t : t + 3 * side;
      const int j_nb = vertical ? (2 - side) + 3 * t : t + 3 * (2 - side);
      D[j_own] = fma(-B, lt[t], D[j_own]);
      E[j_nb] = fma(B, lt[t], E[j_nb]);
    }
  }
  if (inner && live) {
    double* dst = row + block_slot<4>(c, nb, n) * 9;
#pragma unroll
    for (int j = 0; j < 9; ++j) dst[j] = E[j];
  }
}

__global__ void __launch_bounds__(kQ2Threads, 3)
    k_assemble_q2_cube(MeshView m, const __grid_constant__ DevFn fn, ElemRule vol, LineRule fr, double s_in, double s_bnd,
                       double* __restrict__ vals) {
  // A_j, C_j of the current face: [parity][cell][q][2][9]; two buffers, so that one barrier per face is enough
  extern __shared__ __align__(16) double q2_smem[];
  double (*tabs)[kQ2Cells][kQ2MaxFacePts * 2 * 9] = reinterpret_cast<double (*)[kQ2Cells][kQ2MaxFacePts * 2 * 9]>(q2_smem);
  double* stage0 = q2_smem + kQ2TabDoubles;
  const int cs = threadIdx.x / 9, i = threadIdx.x % 9;
  const int k_raw = blockIdx.x * kQ2Cells + cs;
  const bool live = k_raw < m.n_own;
  const int k = live ? k_raw : m.n_own - 1;  // idle threads of the last CTA recompute its last cell (they take part in the barriers)
  const int c = m.own0 + k;
  Geo<HDD_CUBE2D> g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  int nb[4];
  load_neigh<4>(m.neigh, k, nb);
  const int nblk = block_count<4>(nb);
  const int k_first = blockIdx.x * kQ2Cells;
  const int64_t base_blk = __ldg(m.blk_start + k_first);
  double* out = vals + base_blk * 81;
  double* stage = stage0 + stage_pad(out);
  double* row = stage + (__ldg(m.blk_start + k) - base_blk) * 81 + int64_t(i) * nblk * 9;
  const int ai = i % 3, bi = i / 3;
  double D[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) D[j] = 0.0;
  // volume: sum_q w (a K grad phi_j) . grad phi_i with the tensor-product basis
  for (int q = 0; q < vol.n; ++q) {
    double lx[3], dx[3], ly[3], dy[3];
    lagrange2(vol.x[q], lx, dx);
    lagrange2(vol.y[q], ly, dy);
    const double a = expression_at(fn, g.x0 + g.hx * vol.x[q], g.y0 + g.hy * vol.y[q]);
    const double wa = vol.w[q] * g.detj * a;
    const double gxi = wa * pick<3>(dx, ai) * pick<3>(ly, bi) * g.ihx, gyi = wa * pick<3>(lx, ai) * pick<3>(dy, bi) * g.ihy;
    const double cx = K[0] * gxi + K[2] * gyi, cy = K[1] * gxi + K[3] * gyi;  // (K grad phi_j) . grad phi_i = grad phi_j . K^T grad phi_i
#pragma unroll
    for (int b = 0; b < 3; ++b)
#pragma unroll
      for (int a2 = 0; a2 < 3; ++a2)
        D[a2 + 3 * b] = fma(dx[a2] * ly[b] * g.ihx, cx, fma(lx[a2] * dy[b] * g.ihy, cy, D[a2 + 3 * b]));
  }
  q2_face<0>(m, fn, g, K, k, c, nb[0], i, fr, s_in, s_bnd, tabs[0][cs], D, row, nb, live);
  q2_face<1>(m, fn, g, K, k, c, nb[1], i, fr, s_in, s_bnd, tabs[1][cs], D, row, nb, live);
  q2_face<2>(m, fn, g, K, k, c, nb[2], i, fr, s_in, s_bnd, tabs[0][cs], D, row, nb, live);
  q2_face<3>(m, fn, g, K, k, c, nb[3], i, fr, s_in, s_bnd, tabs[1][cs], D, row, nb, live);
  if (live) {
    double* dst = row + block_slot<4>(c, nb, c) * 9;
#pragma unroll
    for (int j = 0; j < 9; ++j) dst[j] = D[j];
  }
  const int k_end = min(k_first + kQ2Cells, m.n_own);
  bulk_write_out(out, stage, (__ldg(m.blk_start + k_end) - base_blk) * 81);
}

// K2 for Q2 on axis-parallel rectangles with a constant or cellwise factor: no quadrature loop at all.  On such a cell every
// integrand of the SWIPDG form is a product of a function of xi and a function of eta, and the quadrature the reference
// prescribes (tensor Gauss rule in the cell, Gauss rule on the faces) sums the two directions independently - so every
// entry is a combination of the entries of five 3 x 3 matrices of the quadratic Lagrange basis on [0,1],
//     M[a][b] = sum_q w_q l_a(t_q) l_b(t_q),   G[a][b] = sum_q w_q l_a(t_q) l_b'(t_q),   S[a][b] = sum_q w_q l_a'(t_q) l_b'(t_q),
// taken with the cell rule's 1-d points (Mv, Gv, Sv: the reference's order-2 rule does not integrate these exactly, which is
// why they are built from the rule and not from the exact integrals) and with the face rule's (Mf, Gf).  With
// phi_j = l_aj(xi) l_bj(eta), j = aj + 3 bj, and for a face: across / along = the 1-d index across / along it,
// u = l_across(face) in {0,1}, v = l_across'(face) / h_across, P = |e| pen (a^- + a^+), Ta = |e| omega^- a^- K^-_nn / h_across,
// Tl = |e| omega^- a^- K^-_nt / h_along (and Ta+, Tl+ with the neighbour's data),
//     en/en  D_ij += Mf[al_i][al_j] (P u_i u_j - Ta (u_i v_j + u_j v_i)) - Tl u_i u_j (Gf[al_i][al_j] + Gf[al_j][al_i])
//     en/ne  E_ij  = Mf[al_i][al_j] (-P u_i u+_j - Ta+ u_i v+_j + Ta v_i u+_j) + u_i u+_j (Tl Gf[al_j][al_i] - Tl+ Gf[al_i][al_j])
// - the sums over the face points of k_assemble_q2_cube's A_j, B_i, C_j carried out by hand.  A row costs ~300 fp64
// operations instead of ~1400, needs no shared-memory tables and no barriers; what is left is the write-out.
struct Q2Tables {
  double Mf[9], Gf[9], Mv[9], Gv[9], Sv[9];
};

static Q2Tables make_q2_tables(const LineRule& vol1d, const LineRule& fr) {
  Q2Tables T{};
  auto fill = [](const LineRule& r, double* M, double* G, double* S) {
    for (int q = 0; q < r.n; ++q) {
      double l[3], d[3];
      lagrange2(r.x[q], l, d);
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) {
          M[3 * a + b] += r.w[q] * l[a] * l[b];
          G[3 * a + b] += r.w[q] * l[a] * d[b];
          if (S) S[3 * a + b] += r.w[q] * d[a] * d[b];
        }
    }
  };
  fill(fr, T.Mf, T.Gf, nullptr);
  fill(vol1d, T.Mv, T.Gv, T.Sv);
  return T;
}

template <int F, int FK>
__device__ __forceinline__ void q2_face_closed(const MeshView& m, const DevFn& fn, const Geo<HDD_CUBE2D>& g, const double* K, int k,
                                               int c, int n, int ai, int bi, double a_self, const Q2Tables& T, double s_in,
                                               double s_bnd, double* D, double* row, const int* nb, bool live) {
  constexpr bool vertical = F < 2;                      // faces 0,1: x = const; faces 2,3: y = const
  constexpr double sgn = (F == 0 || F == 2) ? -1.0 : 1.0;
  constexpr int side = (F == 1 || F == 3) ? 2 : 0;      // 1-d node on the face: own side, the neighbour's is 2 - side
  // l' across the face at the face coordinate (0 or 1) for the own cell and for the neighbour: (-3, 4, -1) or (1, -4, 3)
  constexpr double dl0[3] = {-3.0, 4.0, -1.0}, dl1[3] = {1.0, -4.0, 3.0};
  const bool inner = n >= 0;
  if (!inner && m.btype && __ldg(m.btype + size_t(4) * k + F) != 1) return;  // Neumann face: nothing on the left-hand side
  const int across = vertical ? ai : bi, along = vertical ? bi : ai;
  const double u_i = across == side ? 1.0 : 0.0;
  const double v_i = side == 0 ? pick<3>(dl0, across) : pick<3>(dl1, across);
  const double h = vertical ? fabs(g.hy) : fabs(g.hx);
  const double ih = vertical ? fabs(g.ihy) : fabs(g.ihx);
  const double i_across = vertical ? g.ihx : g.ihy, i_along = vertical ? g.ihy : g.ihx;
  const double kn_ac = sgn * (vertical ? K[0] : K[3]), kn_al = sgn * (vertical ? K[1] : K[2]);
  const double dm = vertical ? K[0] : K[3];
  double wm = 1.0, wp = 0.0, pen0 = s_bnd * dm * ih, a_nb = 0.0, kn_ac_p = 0.0, kn_al_p = 0.0, i_across_p = 0.0;
  if (inner) {
    double Kn[4];
    load_tensor(m.tensor, n, Kn);
    const double dp = vertical ? Kn[0] : Kn[3];
    const double isum = 1.0 / (dp + dm);
    wm = dp * isum;
    wp = dm * isum;
    pen0 = s_in * dp * dm * isum * 0.5 * ih;
    kn_ac_p = sgn * (vertical ? Kn[0] : Kn[3]);
    kn_al_p = sgn * (vertical ? Kn[1] : Kn[2]);
    a_nb = a_self;
    if constexpr (FK == HDD_FN_CELLWISE) a_nb = __ldg(fn.cell + n);
    Geo<HDD_CUBE2D> gn;
    gn.load(m.cgeo, n);
    i_across_p = vertical ? gn.ihx : gn.ihy;
  }
  const double P = h * pen0 * (a_self + a_nb);
  const double cm = h * wm * a_self, cp = h * wp * a_nb;
  const double Ta = cm * i_across * kn_ac, Tl = cm * i_along * kn_al;
  double Mi[3], Gij[3], Gji[3];
#pragma unroll
  for (int b = 0; b < 3; ++b) {
    Mi[b] = T.Mf[along * 3 + b];
    Gij[b] = T.Gf[along * 3 + b];
    Gji[b] = T.Gf[b * 3 + along];
  }
#pragma unroll
  for (int acj = 0; acj < 3; ++acj) {
    const double u_j = acj == side ? 1.0 : 0.0;
    const double v_j = side == 0 ? dl0[acj] : dl1[acj];
    const double cD = P * u_i * u_j - Ta * (u_i * v_j + u_j * v_i);
#pragma unroll
    for (int alj = 0; alj < 3; ++alj) {
      const int j = vertical ? acj + 3 * alj : alj + 3 * acj;
      D[j] = fma(Mi[alj], cD, D[j]);
      if (acj == side) D[j] = fma(-Tl * u_i, Gij[alj] + Gji[alj], D[j]);
    }
  }
  if (!inner) return;
  const double Tap = cp * i_across_p * kn_ac_p, Tlp = cp * i_along * kn_al_p;
  double* dst = row + block_slot<4>(c, nb, n) * 9;
#pragma unroll
  for (int acj = 0; acj < 3; ++acj) {
    const double un_j = acj == 2 - side ? 1.0 : 0.0;
    const double vn_j = side == 0 ? dl1[acj] : dl0[acj];
    const double cE = -P * u_i * un_j - Tap * u_i * vn_j + Ta * v_i * un_j;
#pragma unroll
    for (int alj = 0; alj < 3; ++alj) {
      const int j = vertical ? acj + 3 * alj : alj + 3 * acj;
      double e = Mi[alj] * cE;
      if (acj == 2 - side) e = fma(u_i, Tl * Gji[alj] - Tlp * Gij[alj], e);
      if (live) dst[j] = e;
    }
  }
}

constexpr int kQ2ClosedSmemBytes = (kQ2StageDoubles + 2) * 8;

template <int FK>
__global__ void __launch_bounds__(kQ2Threads, 4)
    k_assemble_q2_closed(MeshView m, const __grid_constant__ DevFn fn, const __grid_constant__ Q2Tables T, double s_in, double s_bnd,
                         double* __restrict__ vals) {
  extern __shared__ __align__(16) double q2_smem[];
  const int cs = threadIdx.x / 9, i = threadIdx.x % 9;
  const int k_raw = blockIdx.x * kQ2Cells + cs;
  const bool live = k_raw < m.n_own;
  const int k = live ? k_raw : m.n_own - 1;  // idle threads of the last CTA recompute its last cell
  const int c = m.own0 + k;
  Geo<HDD_CUBE2D> g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  int nb[4];
  load_neigh<4>(m.neigh, k, nb);
  const int nblk = block_count<4>(nb);
  const int k_first = blockIdx.x * kQ2Cells;
  const int64_t base_blk = __ldg(m.blk_start + k_first);
  double* out = vals + base_blk * 81;
  double* stage = q2_smem + stage_pad(out);
  double* row = stage + (__ldg(m.blk_start + k) - base_blk) * 81 + int64_t(i) * nblk * 9;
  double a_self = fn.value;
  if constexpr (FK == HDD_FN_CELLWISE) a_self = __ldg(fn.cell + c);
  const int ai = i % 3, bi = i / 3;
  // volume: a |T| sum over the four gradient pairings of (1-d matrix in x) x (1-d matrix in y)
  double D[9];
  {
    const double ad = a_self * g.detj;
    const double c0 = ad * K[0] * g.ihx * g.ihx, c1 = ad * K[2] * g.ihx * g.ihy, c2 = ad * K[1] * g.ihx * g.ihy, c3 = ad * K[3] * g.ihy * g.ihy;
    double xS[3], xM[3], xG[3], xGt[3], yS[3], yM[3], yG[3], yGt[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      xS[b] = c0 * T.Sv[ai * 3 + b];
      xM[b] = c3 * T.Mv[ai * 3 + b];
      xG[b] = c1 * T.Gv[ai * 3 + b];   // sum w l_ai l_aj'
      xGt[b] = c2 * T.Gv[b * 3 + ai];  // sum w l_aj l_ai'
      yS[b] = T.Sv[bi * 3 + b];
      yM[b] = T.Mv[bi * 3 + b];
      yG[b] = T.Gv[bi * 3 + b];        // sum w l_bi l_bj'
      yGt[b] = T.Gv[b * 3 + bi];       // sum w l_bj l_bi'
    }
#pragma unroll
    for (int bj = 0; bj < 3; ++bj)
#pragma unroll
      for (int aj = 0; aj < 3; ++aj)
        D[aj + 3 * bj] = fma(xS[aj], yM[bj], fma(xG[aj], yGt[bj], fma(xGt[aj], yG[bj], xM[aj] * yS[bj])));
  }
  q2_face_closed<0, FK>(m, fn, g, K, k, c, nb[0], ai, bi, a_self, T, s_in, s_bnd, D, row, nb, live);
  q2_face_closed<1, FK>(m, fn, g, K, k, c, nb[1], ai, bi, a_self, T, s_in, s_bnd, D, row, nb, live);
  q2_face_closed<2, FK>(m, fn, g, K, k, c, nb[2], ai, bi, a_self, T, s_in, s_bnd, D, row, nb, live);
  q2_face_closed<3, FK>(m, fn, g, K, k, c, nb[3], ai, bi, a_self, T, s_in, s_bnd, D, row, nb, live);
  if (live) {
    double* dst = row + block_slot<4>(c, nb, c) * 9;
#pragma unroll
    for (int j = 0; j < 9; ++j) dst[j] = D[j];
  }
  const int k_end = min(k_first + kQ2Cells, m.n_own);
  bulk_write_out(out, stage, (__ldg(m.blk_start + k_end) - base_blk) * 81);
}

// Volume-pattern products (discretizations/swipdg.hh:359-443): one dense n_loc x n_loc block per cell, one thread per
// row.  WHICH 0 "l2" int phi_i phi_j, 1 "h1_semi" int grad phi_j . grad phi_i, 2 "elliptic" int a K grad phi_j . grad
// phi_i, 3 "boundary_l2" int_{dT on dOmega} phi_i phi_j.  over_integrate = 2 is folded into the rules by the launcher.
template <int KIND, int P, int WHICH>
__global__ void __launch_bounds__(kThreads)
    k_assemble_block_product(MeshView m, const __grid_constant__ DevFn fn, ElemRule vol, LineRule fr,
                             double* __restrict__ vals) {
  using G = Elem<KIND, P>;
  constexpr int NL = G::NL, NF = G::NF;
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= int64_t(m.n_own) * NL) return;
  const int k = int(t / NL), i = int(t % NL);
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double D[NL];
#pragma unroll
  for (int j = 0; j < NL; ++j) D[j] = 0.0;
  if constexpr (WHICH <= 2) {
    double K[4] = {1.0, 0.0, 0.0, 1.0};
    if constexpr (WHICH == 2) load_tensor(m.tensor, c, K);
    for (int q = 0; q < vol.n; ++q) {
      double phi[NL], gx[NL], gy[NL], x, y;
      g.basis(vol.x[q], vol.y[q], phi, gx, gy);
      g.to_global(vol.x[q], vol.y[q], x, y);
      double w = vol.w[q] * g.detj;
      if constexpr (WHICH == 2) w *= fn_eval(fn, c, x, y);
      if constexpr (WHICH == 0) {
        const double pi = w * pick<NL>(phi, i);
#pragma unroll
        for (int j = 0; j < NL; ++j) D[j] = fma(pi, phi[j], D[j]);
      } else {
        const double gxi = w * pick<NL>(gx, i), gyi = w * pick<NL>(gy, i);
#pragma unroll
        for (int j = 0; j < NL; ++j)
          D[j] = fma(K[0] * gx[j] + K[1] * gy[j], gxi, fma(K[2] * gx[j] + K[3] * gy[j], gyi, D[j]));
      }
    }
  } else {
    int nb[NF];
    load_neigh<NF>(m.neigh, k, nb);
#pragma unroll 1
    for (int f = 0; f < NF; ++f) {
      if (nb[f] >= 0) continue;
      const FaceGeo e = make_face(g, f);
      for (int q = 0; q < fr.n; ++q) {
        const double x = e.ax + fr.x[q] * (e.bx - e.ax), y = e.ay + fr.x[q] * (e.by - e.ay);
        double xi, eta, phi[NL], gx[NL], gy[NL];
        g.to_local(x, y, xi, eta);
        g.basis(xi, eta, phi, gx, gy);
        const double pi = fr.w[q] * e.h * pick<NL>(phi, i);
#pragma unroll
        for (int j = 0; j < NL; ++j) D[j] = fma(pi, phi[j], D[j]);
      }
    }
  }
  double* dst = vals + size_t(t) * NL;
#pragma unroll
  for (int j = 0; j < NL; ++j) dst[j] = D[j];
}

// K3a.  Functionals::L2Volume(force) (discretizations/swipdg.hh:253-271): rule of order(f) + p.
// TRIG: the force is c cos(..) cos(..) of affine arguments (TrigProduct, expr.hpp): the reference-to-cell map of both cell
// types is affine, so per cell the arguments are affine in (xi, eta) and a point costs two fast_cos instead of the general
// function evaluation (see k_indicators).
template <int KIND, int P, bool TRIG>
__global__ void __launch_bounds__(kThreads)
    k_rhs_volume(MeshView m, const __grid_constant__ DevFn fn, const __grid_constant__ TrigProduct tp, ElemRule vol, int accumulate,
                 double* __restrict__ b) {
  using G = Elem<KIND, P>;
  constexpr int NL = G::NL;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double acc[NL];
#pragma unroll
  for (int i = 0; i < NL; ++i) acc[i] = 0.0;
  double t00 = 0.0, t0x = 0.0, t0y = 0.0, t10 = 0.0, t1x = 0.0, t1y = 0.0;
  bool trig = false;
  if (TRIG) {
    double ox, oy, px, py, qx, qy;
    g.to_global(0.0, 0.0, ox, oy);
    g.to_global(1.0, 0.0, px, py);
    g.to_global(0.0, 1.0, qx, qy);
    t00 = fma(tp.a[0], ox, fma(tp.b[0], oy, tp.d[0]));
    t0x = tp.a[0] * (px - ox) + tp.b[0] * (py - oy);
    t0y = tp.a[0] * (qx - ox) + tp.b[0] * (qy - oy);
    t10 = fma(tp.a[1], ox, fma(tp.b[1], oy, tp.d[1]));
    t1x = tp.a[1] * (px - ox) + tp.b[1] * (py - oy);
    t1y = tp.a[1] * (qx - ox) + tp.b[1] * (qy - oy);
    trig = fabs(t00) + fabs(t0x) + fabs(t0y) < kFastCosMax && fabs(t10) + fabs(t1x) + fabs(t1y) < kFastCosMax;
  }
  for (int q = 0; q < vol.n; ++q) {
    double phi[NL], gx[NL], gy[NL], x, y;
    g.basis(vol.x[q], vol.y[q], phi, gx, gy);
    double fv;
    if (TRIG && trig) {
      fv = tp.c * fast_cos(fma(t0x, vol.x[q], fma(t0y, vol.y[q], t00))) * fast_cos(fma(t1x, vol.x[q], fma(t1y, vol.y[q], t10)));
    } else {
      g.to_global(vol.x[q], vol.y[q], x, y);
      fv = fn_eval(fn, c, x, y);
    }
    fv *= vol.w[q] * g.detj;
#pragma unroll
    for (int i = 0; i < NL; ++i) acc[i] += fv * phi[i];
  }
#pragma unroll
  for (int i = 0; i < NL; ++i) b[size_t(NL) * k + i] = accumulate ? b[size_t(NL) * k + i] + acc[i] : acc[i];
}

// K3a', Q1 on axis-parallel cells with a separable force f(x,y) = g(x) h(y): the tensor Gauss rule needs only
// n + n evaluations of the (transcendental) factors per cell instead of n * n of the full expression.
__global__ void __launch_bounds__(kThreads)
    k_rhs_volume_cube_separable(MeshView m, const __grid_constant__ DevFn fn, LineRule g1, int accumulate,
                                double* __restrict__ b) {
  using G = Geo<HDD_CUBE2D>;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double fx[kMaxLinePts], fy[kMaxLinePts];
  for (int i = 0; i < g1.n; ++i) {
    const double vx[2] = {g.x0 + g.hx * g1.x[i], 0.0}, vy[2] = {0.0, g.y0 + g.hy * g1.x[i]};
    fx[i] = eval_program(fn.px, vx) * g1.w[i];
    fy[i] = eval_program(fn.py, vy) * g1.w[i];
  }
  // b_i = detj * sum_{q,r} w_q w_r g(x_q) h(y_r) phi_i(xi_q, xi_r), phi tensor: (1-xi | xi) x (1-eta | eta)
  double sx0 = 0.0, sx1 = 0.0, sy0 = 0.0, sy1 = 0.0;
  for (int i = 0; i < g1.n; ++i) {
    sx0 = fma(fx[i], 1.0 - g1.x[i], sx0); sx1 = fma(fx[i], g1.x[i], sx1);
    sy0 = fma(fy[i], 1.0 - g1.x[i], sy0); sy1 = fma(fy[i], g1.x[i], sy1);
  }
  double* dst = b + size_t(4) * k;
  double o0 = g.detj * sx0 * sy0, o1 = g.detj * sx1 * sy0, o2 = g.detj * sx0 * sy1, o3 = g.detj * sx1 * sy1;
  if (accumulate) { o0 += dst[0]; o1 += dst[1]; o2 += dst[2]; o3 += dst[3]; }
  asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst), "d"(o0), "d"(o1), "d"(o2), "d"(o3) : "memory");
}

// K3a'', tensor-product grid + separable force f = g(x) h(y): the one-dimensional moments
//   SX[cx][a] = h_x sum_q w_q g(x_q) l_a(xi_q),  SY[cy][b] = h_y sum_q w_q h(y_q) l_b(eta_q)
// depend on the column / row of the cell only, so they are evaluated once per column and row (nx + ny instead of
// nx * ny evaluations of the transcendental factors) and the cell kernel is a pure stream: b_(a + (p+1) b) = SX_a SY_b.
// The column / row geometry comes from MeshView::tgeo.
template <int P>
__global__ void k_rhs_tensor_moments(const __grid_constant__ DevFn fn, LineRule g1, int nx, int ny,
                                     const double* __restrict__ geo, double* __restrict__ mom) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nx + ny) return;
  const bool is_x = t < nx;
  const double2 oh = reinterpret_cast<const double2*>(geo)[2 * size_t(t)];  // {origin, size} of column / row t
  double acc[P + 1];
#pragma unroll
  for (int a = 0; a <= P; ++a) acc[a] = 0.0;
  for (int q = 0; q < g1.n; ++q) {
    const double xi = g1.x[q];
    const double pos = oh.x + oh.y * xi;
    const double v[2] = {is_x ? pos : 0.0, is_x ? 0.0 : pos};
    const double f = eval_program(is_x ? fn.px : fn.py, v) * g1.w[q];
    if constexpr (P == 1) {
      acc[0] = fma(f, 1.0 - xi, acc[0]);
      acc[1] = fma(f, xi, acc[1]);
    } else {
      acc[0] = fma(f, (1.0 - xi) * (1.0 - 2.0 * xi), acc[0]);
      acc[1] = fma(f, 4.0 * xi * (1.0 - xi), acc[1]);
      acc[2] = fma(f, xi * (2.0 * xi - 1.0), acc[2]);
    }
  }
#pragma unroll
  for (int a = 0; a <= P; ++a) mom[size_t(t) * (P + 1) + a] = fabs(oh.y) * acc[a];
}

template <int P>
__global__ void __launch_bounds__(256)
    k_rhs_tensor_cells(int32_t n_own, int32_t own0, const int32_t* __restrict__ cell_v0, int nx,
                       const double* __restrict__ mom, int accumulate, double* __restrict__ b) {
  constexpr int N1 = P + 1, NL = N1 * N1;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_own) return;
  const int v0 = __ldg(cell_v0 + own0 + k);
  const int cx = v0 % (nx + 1), cy = v0 / (nx + 1);
  double sx[N1], sy[N1];
#pragma unroll
  for (int a = 0; a < N1; ++a) {
    sx[a] = __ldg(mom + size_t(cx) * N1 + a);
    sy[a] = __ldg(mom + size_t(nx + cy) * N1 + a);
  }
  double* dst = b + size_t(NL) * k;
  if constexpr (P == 1) {
    double o0 = sx[0] * sy[0], o1 = sx[1] * sy[0], o2 = sx[0] * sy[1], o3 = sx[1] * sy[1];
    if (accumulate) { o0 += dst[0]; o1 += dst[1]; o2 += dst[2]; o3 += dst[3]; }
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst), "d"(o0), "d"(o1), "d"(o2), "d"(o3) : "memory");
  } else {
#pragma unroll
    for (int bb = 0; bb < N1; ++bb)
#pragma unroll
      for (int a = 0; a < N1; ++a) {
        const double o = sx[a] * sy[bb];
        dst[a + N1 * bb] = accumulate ? dst[a + N1 * bb] + o : o;
      }
  }
}

// K3b.  Functionals::DirichletBoundarySWIPDG (discretizations/swipdg.hh:273-332; SWIPDG::BoundaryRHS):
// b_i += int_e -g (A grad phi_i . n) + pen g phi_i
template <int KIND, int P>
__global__ void __launch_bounds__(kThreads)
    k_rhs_dirichlet(MeshView m, const __grid_constant__ DevFn fac, const __grid_constant__ DevFn dir, LineRule fr,
                    double s_bnd, double* __restrict__ b) {
  using G = Elem<KIND, P>;
  constexpr int NL = G::NL, NF = G::NF;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  const int c = m.own0 + k;
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  bool any = false;
#pragma unroll
  for (int f = 0; f < NF; ++f) any |= nb[f] < 0;
  if (!any) return;
  G g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  double acc[NL];
#pragma unroll
  for (int i = 0; i < NL; ++i) acc[i] = 0.0;
  for (int f = 0; f < NF; ++f) {
    if (nb[f] >= 0) continue;
    if (m.btype && __ldg(m.btype + size_t(NF) * k + f) != 1) continue;
    const FaceGeo e = make_face(g, f);
    const double dm = e.nx * (K[0] * e.nx + K[1] * e.ny) + e.ny * (K[2] * e.nx + K[3] * e.ny);
    for (int q = 0; q < fr.n; ++q) {
      const double x = e.ax + fr.x[q] * (e.bx - e.ax), y = e.ay + fr.x[q] * (e.by - e.ay);
      double xi, eta, phi[NL], gx[NL], gy[NL];
      g.to_local(x, y, xi, eta);
      g.basis(xi, eta, phi, gx, gy);
      const double a = fn_eval(fac, c, x, y), gd = fn_eval(dir, c, x, y);
      const double pen = s_bnd * dm * a / e.h;
      const double w = fr.w[q] * e.h;
#pragma unroll
      for (int i = 0; i < NL; ++i) {
        const double fl = a * ((K[0] * gx[i] + K[1] * gy[i]) * e.nx + (K[2] * gx[i] + K[3] * gy[i]) * e.ny);
        acc[i] += w * (-gd * fl + pen * gd * phi[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NL; ++i) b[size_t(NL) * k + i] += acc[i];
}

// K3c.  Functionals::L2Face(neumann) on the Neumann faces (discretizations/swipdg.hh:335-356): b_i += int_e g_N phi_i
template <int KIND, int P>
__global__ void __launch_bounds__(kThreads)
    k_rhs_neumann(MeshView m, const __grid_constant__ DevFn neu, LineRule fr, double* __restrict__ b) {
  using G = Elem<KIND, P>;
  constexpr int NL = G::NL, NF = G::NF;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own || !m.btype) return;
  const int c = m.own0 + k;
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  bool any = false;
#pragma unroll
  for (int f = 0; f < NF; ++f) any |= nb[f] < 0 && __ldg(m.btype + size_t(NF) * k + f) == 2;
  if (!any) return;
  G g;
  g.load(m.cgeo, c);
  double acc[NL];
#pragma unroll
  for (int i = 0; i < NL; ++i) acc[i] = 0.0;
  for (int f = 0; f < NF; ++f) {
    if (nb[f] >= 0 || __ldg(m.btype + size_t(NF) * k + f) != 2) continue;
    const FaceGeo e = make_face(g, f);
    for (int q = 0; q < fr.n; ++q) {
      const double x = e.ax + fr.x[q] * (e.bx - e.ax), y = e.ay + fr.x[q] * (e.by - e.ay);
      double xi, eta, phi[NL], gx[NL], gy[NL];
      g.to_local(x, y, xi, eta);
      g.basis(xi, eta, phi, gx, gy);
      const double gn = fn_eval(neu, c, x, y) * fr.w[q] * e.h;
#pragma unroll
      for (int i = 0; i < NL; ++i) acc[i] = fma(gn, phi[i], acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < NL; ++i) b[size_t(NL) * k + i] += acc[i];
}

// K4.  out = sum_k theta_k part_k, 256-bit streaming loads/stores.
__global__ void __launch_bounds__(256) k_freeze(FreezeArgs a, double* __restrict__ out, int64_t count) {
  const int64_t n4 = count / 4;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
    for (int k = 0; k < a.n; ++k) {
      double v0, v1, v2, v3;
      asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                   : "=d"(v0), "=d"(v1), "=d"(v2), "=d"(v3)
                   : "l"(a.part[k] + 4 * i));
      s0 += a.theta[k] * v0; s1 += a.theta[k] * v1; s2 += a.theta[k] * v2; s3 += a.theta[k] * v3;
    }
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(out + 4 * i), "d"(s0), "d"(s1), "d"(s2), "d"(s3) : "memory");
  }
  for (int64_t i = 4 * n4 + int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride) {
    double s = 0;
    for (int k = 0; k < a.n; ++k) s += a.theta[k] * a.part[k][i];
    out[i] = s;
  }
}

template <int NF, int NL>
__global__ void k_extract_dinv(MeshView m, const double* __restrict__ values, int jacobi,
                               double* __restrict__ dinv) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= int64_t(m.n_own) * NL) return;
  if (!jacobi) { dinv[t] = 1.0; return; }
  const int k = int(t / NL), i = int(t % NL);
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  const int self = m.own0 + k;
  const int nblk = block_count<NF>(nb);
  const int slot = block_slot<NF>(self, nb, self);
  const double d = values[m.blk_start[k] * (NL * NL) + int64_t(i) * nblk * NL + slot * NL + i];
  dinv[t] = 1.0 / d;
}

}  // namespace

void launch_build_geometry(int kind, int32_t n_loc, int32_t v_begin, int32_t v_end, const double* xy, const int32_t* cell_verts_local,
                           double* cgeo, int32_t* flag, cudaStream_t s) {
  if (n_loc == 0) return;
  k_build_geometry<<<grid_for(n_loc, 256), 256, 0, s>>>(kind, n_loc, v_begin, v_end, xy, cell_verts_local, cgeo, flag);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_cube_fill(const CubeGridDesc& g, int32_t n_loc, int32_t own0, int32_t n_own, int32_t cell_begin, const int32_t* halo,
                      double* cgeo, int32_t* cell_v0, int32_t* lex_cell, int32_t* cgid, int32_t* neigh, double* tgeo,
                      cudaStream_t s) {
  if (n_loc > 0)
    k_cube_fill<<<grid_for(n_loc, 256), 256, 0, s>>>(g, n_loc, own0, n_own, cell_begin, halo, cgeo, cell_v0, lex_cell, cgid, neigh);
  k_cube_tgeo<<<grid_for(g.nx + g.ny, 256), 256, 0, s>>>(g, tgeo);
  count_launch(2);
  HDD_CUDA(cudaGetLastError());
}

void launch_validate_neighbours(const int32_t* neigh, int64_t count, int32_t n_cells, int32_t* flag, cudaStream_t s) {
  if (count == 0) return;
  k_validate_neighbours<<<grid_for(count, 256), 256, 0, s>>>(neigh, count, n_cells, flag);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_iota(int32_t* out, int32_t n, cudaStream_t s) {
  if (n == 0) return;
  k_iota<<<grid_for(n, 256), 256, 0, s>>>(out, n, 0);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_iota_from(int32_t* out, int32_t n, int32_t first, cudaStream_t s) {
  if (n == 0) return;
  k_iota<<<grid_for(n, 256), 256, 0, s>>>(out, n, first);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_subdomain_structure(const int32_t* sub, const int32_t* neigh, int nf, int32_t n_cells, int n_sub,
                                int64_t* offsets, uint8_t* adj, int32_t* flag, cudaStream_t s) {
  k_subdomain_structure<<<grid_for(n_cells, 256), 256, 0, s>>>(sub, neigh, nf, n_cells, n_sub, offsets, adj, flag);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_localize_neighbours(int32_t* neigh, int64_t count, int32_t cell_begin, int32_t cell_end, const int32_t* halo,
                                int32_t n_lo, int32_t n_hi, int32_t* flag, cudaStream_t s) {
  if (count == 0) return;
  k_localize_neighbours<<<grid_for(count, 256), 256, 0, s>>>(neigh, count, cell_begin, cell_end, halo, n_lo, n_hi, flag);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_count_blocks(const MeshView& m, int64_t* nblk, cudaStream_t s) {
  if (m.n_own == 0) return;
  k_count_blocks<<<grid_for(m.n_own, 256), 256, 0, s>>>(m, nblk);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void exclusive_scan_i64(const int64_t* in, int64_t* out, int64_t n, cudaStream_t s) {
  size_t bytes = 0;
  HDD_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, int(n), s));
  // scratch from the library's caching allocator: the stream-ordered allocator (cudaMallocAsync) grows and trims its pool
  // at synchronisation points, and with peer access enabled a fresh block is mapped on every peer - measured as sporadic
  // 10-190 ms stalls of this call on 2 ranks
  DevBuf<unsigned char> tmp;
  tmp.alloc(bytes > 0 ? bytes : 1);
  HDD_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, bytes, in, out, int(n), s));
  HDD_CUDA(cudaStreamSynchronize(s));  // the scratch goes back to the cache when tmp leaves scope
  count_launch(2);
}

// compile-time dispatch helpers: (element kind, polynomial order) and factor kind
template <class F>
static void dispatch_elem(int kind, int polorder, F&& f) {
  if (polorder != 1 && polorder != 2) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "polorder " << polorder);
  if (kind == HDD_SIMPLEX2D) {
    if (polorder == 1) f(ic<HDD_SIMPLEX2D>{}, ic<1>{}); else f(ic<HDD_SIMPLEX2D>{}, ic<2>{});
  } else {
    if (polorder == 1) f(ic<HDD_CUBE2D>{}, ic<1>{}); else f(ic<HDD_CUBE2D>{}, ic<2>{});
  }
}

template <class F>
static void dispatch_fk(int fk, F&& f) {
  if (fk == HDD_FN_CONSTANT) f(ic<HDD_FN_CONSTANT>{});
  else if (fk == HDD_FN_CELLWISE) f(ic<HDD_FN_CELLWISE>{});
  else f(ic<HDD_FN_EXPRESSION>{});
}

void launch_fill_csr(const MeshView& m, int64_t* rowptr, int32_t* col, cudaStream_t s) {
  if (m.n_own == 0) return;
  const int64_t rows = int64_t(m.n_own) * m.nl;
  dispatch_block(m, [&](auto nf, auto nl) {
    k_fill_csr<decltype(nf)::value, decltype(nl)::value><<<grid_for(rows, 256), 256, 0, s>>>(m, rowptr, col);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

// The left-hand-side kernel for (grid, polOrder, factor kind); "closed" = a factor constant per cell (constant or cell-wise):
//   P1 triangles   closed: k_assemble_p1_closed<FK>   Expression: k_assemble_lhs
//   Q1 rectangles  k_assemble_lhs_cube<FK, 4, true> with the tensor-grid tables (m.tgeo), else <FK, 3, false>
//   Q2 rectangles  closed: k_assemble_q2_closed<FK>   Expression: k_assemble_q2_cube for up to kQ2MaxFacePts face points,
//                  else k_assemble_rows
//   P2 triangles   k_assemble_rows<FK>
void launch_assemble_lhs(const MeshView& m, const DevFn& factor_dev, int factor_kind, int factor_order, int polorder,
                         double* values, cudaStream_t s) {
  if (m.n_own == 0) return;
  if (polorder != 1 && polorder != 2) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "polorder " << polorder);
  const ElemRule vol = element_rule(m.kind, factor_order + 2 * (polorder - 1));
  const LineRule fr = line_rule(factor_order + 2 * polorder);
  const double si = sigma_inner(polorder), sb = sigma_boundary(polorder);
  const int blocks = grid_for(m.n_own, kThreads);
  // p = 2 row kernel: one thread per row, 3 CTAs per SM (168 registers; 2.85 ms vs 3.48 ms with 2 at 1024^2 Q2)
  const int row_blocks = grid_for(int64_t(m.n_own) * m.nl, kThreads);
  if (m.kind == HDD_SIMPLEX2D && polorder == 1) {
    if (factor_kind == HDD_FN_CONSTANT)
      k_assemble_p1_closed<HDD_FN_CONSTANT><<<blocks, kThreads, 0, s>>>(m, factor_dev, si, sb, values);
    else if (factor_kind == HDD_FN_CELLWISE)
      k_assemble_p1_closed<HDD_FN_CELLWISE><<<blocks, kThreads, 0, s>>>(m, factor_dev, si, sb, values);
    else
      k_assemble_lhs<<<blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, si, sb, values);
  } else if (polorder == 1) {
    // resident CTAs per SM the kernel is compiled for: 3 (160 registers) for the general kernel, 4 (128) for the tensor
    // grid variant, which keeps no neighbour geometry records alive (measured 2.15 -> 2.03 ms at 4096^2; 5 CTAs spill:
    // 2.81 ms)
    // (closed-form entries as in the P1 / Q2 kernels were tried here as well - half the fp64 work, 40 % fewer instructions,
    // 5 resident CTAs: 2.07 ms against 2.05-2.09 ms, and 2.37 ms when a thread stores row after row instead of block after
    // block - this kernel is limited by its scattered 32-byte-sector store stream, not by instruction issue; DESIGN.md 4)
    dispatch_fk(factor_kind, [&](auto k) {
      constexpr int FK = decltype(k)::value;
      if (m.tgeo)
        k_assemble_lhs_cube<FK, 4, true><<<blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, si, sb, values);
      else
        k_assemble_lhs_cube<FK, 3, false><<<blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, si, sb, values);
    });
  } else if (m.kind == HDD_CUBE2D) {
    const int q2_blocks = (m.n_own + kQ2Cells - 1) / kQ2Cells;
    if (factor_kind != HDD_FN_EXPRESSION) {
      const Q2Tables T = make_q2_tables(line_rule(factor_order + 2 * (polorder - 1)), fr);
      auto launch = [&](auto kern) {
        HDD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kQ2ClosedSmemBytes));
        kern<<<q2_blocks, kQ2Threads, kQ2ClosedSmemBytes, s>>>(m, factor_dev, T, si, sb, values);
      };
      if (factor_kind == HDD_FN_CONSTANT) launch(k_assemble_q2_closed<HDD_FN_CONSTANT>);
      else launch(k_assemble_q2_closed<HDD_FN_CELLWISE>);
    } else if (fr.n <= kQ2MaxFacePts) {
      HDD_CUDA(cudaFuncSetAttribute(k_assemble_q2_cube, cudaFuncAttributeMaxDynamicSharedMemorySize, kQ2SmemBytes));
      k_assemble_q2_cube<<<q2_blocks, kQ2Threads, kQ2SmemBytes, s>>>(m, factor_dev, vol, fr, si, sb, values);
    } else {
      k_assemble_rows<HDD_CUBE2D, 2, HDD_FN_EXPRESSION, 0, 3>
          <<<row_blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, si, sb, values);
    }
  } else {
    dispatch_fk(factor_kind, [&](auto k) {
      k_assemble_rows<HDD_SIMPLEX2D, 2, decltype(k)::value, 0, 3>
          <<<row_blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, si, sb, values);
    });
  }
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

// over_integrate of the product assemblers (discretizations/swipdg.hh:359, block-swipdg.hh:399)
constexpr int kOverIntegrate = 2;

void launch_assemble_penalty(const MeshView& m, const DevFn& factor_dev, int factor_kind, int factor_order, int polorder,
                             double* values, cudaStream_t s) {
  if (m.n_own == 0) return;
  const ElemRule vol = element_rule(m.kind, 0);  // unused
  const LineRule fr = line_rule(factor_order + 2 * polorder + kOverIntegrate);
  const double si = sigma_inner(polorder), sb = sigma_boundary(polorder);
  const int64_t rows = int64_t(m.n_own) * m.nl;
  dispatch_elem(m.kind, polorder, [&](auto kind, auto p) {
    dispatch_fk(factor_kind, [&](auto k) {
      k_assemble_rows<decltype(kind)::value, decltype(p)::value, decltype(k)::value, 1>
          <<<grid_for(rows, kThreads), kThreads, 0, s>>>(m, factor_dev, vol, fr, si, sb, values);
    });
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_assemble_block_product(const MeshView& m, int which, const DevFn& factor_dev, int factor_order, int polorder,
                                   double* values, cudaStream_t s) {
  if (m.n_own == 0) return;
  const int p = polorder;
  const int vorder = which == 0 ? 2 * p + kOverIntegrate
                                : which == 1 ? 2 * (p - 1) + kOverIntegrate : factor_order + 2 * (p - 1) + kOverIntegrate;
  const ElemRule vol = element_rule(m.kind, vorder);
  const LineRule fr = line_rule(2 * p + kOverIntegrate);
  const int64_t rows = int64_t(m.n_own) * m.nl;
  const int blocks = grid_for(rows, kThreads);
  dispatch_elem(m.kind, polorder, [&](auto kind, auto pp) {
    constexpr int KD = decltype(kind)::value, PP = decltype(pp)::value;
    switch (which) {
      case 0: k_assemble_block_product<KD, PP, 0><<<blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, values); break;
      case 1: k_assemble_block_product<KD, PP, 1><<<blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, values); break;
      case 2: k_assemble_block_product<KD, PP, 2><<<blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, values); break;
      case 3: k_assemble_block_product<KD, PP, 3><<<blocks, kThreads, 0, s>>>(m, factor_dev, vol, fr, values); break;
      default: HDD_THROW(HDD_ERR_INTERNAL, "unknown block product " << which);
    }
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_rhs_volume(const MeshView& m, const DevFn& force_dev, int force_order, bool separable, int polorder,
                       bool accumulate, const TensorGridView* tg, double* b, cudaStream_t s) {
  if (m.n_own == 0) return;
  const int acc = accumulate ? 1 : 0;
  if (m.kind == HDD_CUBE2D && separable && tg && tg->nx > 0 && tg->scratch && m.tgeo) {
    // tensor-product grid: 1-d moments per column / row, then a pure streaming kernel
    const LineRule g1 = line_rule(force_order + polorder);
    const int nx = tg->nx, ny = tg->ny, n1 = polorder + 1;
    const double* geo = m.tgeo;  // {x0, hx} per column, {y0, hy} per row (built at mesh creation)
    double* mom = tg->scratch;   // [(nx + ny) * (p + 1)]
    if (polorder == 1) {
      k_rhs_tensor_moments<1><<<grid_for(nx + ny, 128), 128, 0, s>>>(force_dev, g1, nx, ny, geo, mom);
      k_rhs_tensor_cells<1><<<grid_for(m.n_own, 256), 256, 0, s>>>(m.n_own, m.own0, tg->cell_v0, nx, mom, acc, b);
    } else {
      k_rhs_tensor_moments<2><<<grid_for(nx + ny, 128), 128, 0, s>>>(force_dev, g1, nx, ny, geo, mom);
      k_rhs_tensor_cells<2><<<grid_for(m.n_own, 256), 256, 0, s>>>(m.n_own, m.own0, tg->cell_v0, nx, mom, acc, b);
    }
    (void)n1;
    count_launch(2);
    HDD_CUDA(cudaGetLastError());
    return;
  }
  if (m.kind == HDD_CUBE2D && separable && polorder == 1) {
    k_rhs_volume_cube_separable<<<grid_for(m.n_own, kThreads), kThreads, 0, s>>>(m, force_dev, line_rule(force_order + polorder), acc, b);
    count_launch();
    HDD_CUDA(cudaGetLastError());
    return;
  }
  const ElemRule vol = element_rule(m.kind, force_order + polorder);
  TrigProduct tp{};
  if (force_dev.kind == HDD_FN_EXPRESSION && force_dev.fast.n_terms > 0) tp = as_trig_product(force_dev.fast);
  dispatch_elem(m.kind, polorder, [&](auto kind, auto p) {
    if (tp.valid)
      k_rhs_volume<decltype(kind)::value, decltype(p)::value, true><<<grid_for(m.n_own, kThreads), kThreads, 0, s>>>(m, force_dev, tp, vol, acc, b);
    else
      k_rhs_volume<decltype(kind)::value, decltype(p)::value, false><<<grid_for(m.n_own, kThreads), kThreads, 0, s>>>(m, force_dev, tp, vol, acc, b);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_rhs_dirichlet(const MeshView& m, const DevFn& factor_dev, int factor_order, const DevFn& dirichlet_dev,
                          int dirichlet_order, int polorder, double* b, cudaStream_t s) {
  if (m.n_own == 0) return;
  const LineRule fr = line_rule(factor_order + dirichlet_order + 2 * polorder);
  const double sb = sigma_boundary(polorder);
  dispatch_elem(m.kind, polorder, [&](auto kind, auto p) {
    k_rhs_dirichlet<decltype(kind)::value, decltype(p)::value>
        <<<grid_for(m.n_own, kThreads), kThreads, 0, s>>>(m, factor_dev, dirichlet_dev, fr, sb, b);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_rhs_neumann(const MeshView& m, const DevFn& neumann_dev, int neumann_order, int polorder, double* b,
                        cudaStream_t s) {
  if (m.n_own == 0 || !m.btype) return;
  const LineRule fr = line_rule(neumann_order + polorder);
  dispatch_elem(m.kind, polorder, [&](auto kind, auto p) {
    k_rhs_neumann<decltype(kind)::value, decltype(p)::value><<<grid_for(m.n_own, kThreads), kThreads, 0, s>>>(m, neumann_dev, fr, b);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_freeze(const FreezeArgs& a, double* out, int64_t count, cudaStream_t s) {
  if (count == 0) return;
  const int blocks = int(std::min<int64_t>((count / 4 + 255) / 256 + 1, 148 * 16));
  k_freeze<<<blocks, 256, 0, s>>>(a, out, count);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_extract_dinv(const MeshView& m, const double* values, int jacobi, double* dinv, cudaStream_t s) {
  if (m.n_own == 0) return;
  const int64_t rows = int64_t(m.n_own) * m.nl;
  dispatch_block(m, [&](auto nf, auto nl) {
    k_extract_dinv<decltype(nf)::value, decltype(nl)::value><<<grid_for(rows, 256), 256, 0, s>>>(m, values, jacobi, dinv);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

}  // namespace hdd
