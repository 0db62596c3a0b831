// K12/K13 for sm_100a: what the reference's product matrices are used for - bilinear forms u^T P v and the induced
// norms (discretizations/base.hh:272-291; test/linearelliptic-swipdg.hh:267-290) - plus the per-cell error norms of
// u_h against an analytic solution (SURVEY 8f rank 3).  All HBM-bound streaming work.
#include "kernels.hpp"

namespace hdd {

namespace {

constexpr int kThreads = 256;

// volume pattern: one dense NL x NL block per owned cell, global column indices
template <int NL>
__global__ void k_fill_volume_csr(MeshView m, int64_t* __restrict__ rowptr, int32_t* __restrict__ col) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t rows = int64_t(m.n_own) * NL;
  if (t > rows) return;
  rowptr[t] = t * NL;
  if (t == rows) return;
  const int k = int(t / NL);
  const int g = __ldg(m.cgid + m.own0 + k);
#pragma unroll
  for (int j = 0; j < NL; ++j) col[t * NL + j] = NL * g + j;
}

// y = P x for a block-diagonal (volume pattern) matrix; x, y over the owned rows
template <int NL>
__global__ void __launch_bounds__(kThreads)
    k_block_spmv(int64_t rows, const double* __restrict__ vals, const double* __restrict__ x, double* __restrict__ y) {
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < rows; t += stride) {
    const double* a = vals + t * NL;
    const double* xs = x + (t / NL) * NL;
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < NL; ++j) s = fma(__ldg(a + j), __ldg(xs + j), s);
    y[t] = s;
  }
}

// K13.  Per owned cell: int_T (u_h - u)^2, int_T |grad(u_h - u)|^2, int_T a K grad(u_h - u).grad(u_h - u)
// (Products::L2 / H1Semi / Elliptic induced norms of the difference, test/linearelliptic-swipdg.hh:267-290), one thread
// per cell, u and its gradient given as expression programs.
template <int KIND, int P>
__global__ void __launch_bounds__(128)
    k_error_norms(MeshView m, const __grid_constant__ DevFn exact, const __grid_constant__ DevFn exact_dx,
                  const __grid_constant__ DevFn exact_dy, const __grid_constant__ DevCombo factor,
                  const DevFn* __restrict__ fn_table, ElemRule rule, const double* __restrict__ u_own,
                  double* __restrict__ out) {
  using G = Elem<KIND, P>;
  constexpr int NL = G::NL;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  double u[NL];
#pragma unroll
  for (int i = 0; i < NL; ++i) u[i] = u_own[size_t(NL) * k + i];
  double l2 = 0.0, h1 = 0.0, en = 0.0;
  for (int q = 0; q < rule.n; ++q) {
    double phi[NL], gx[NL], gy[NL], x, y;
    g.basis(rule.x[q], rule.y[q], phi, gx, gy);
    g.to_global(rule.x[q], rule.y[q], x, y);
    double uv = 0.0, ux = 0.0, uy = 0.0;
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      uv = fma(u[i], phi[i], uv);
      ux = fma(u[i], gx[i], ux);
      uy = fma(u[i], gy[i], uy);
    }
    const double d = uv - fn_eval(exact, c, x, y), ex = ux - fn_eval(exact_dx, c, x, y), ey = uy - fn_eval(exact_dy, c, x, y);
    const double w = rule.w[q] * g.detj;
    const double a = factor.n > 0 ? combo_eval(factor, fn_table, c, x, y) : 1.0;
    l2 = fma(w * d, d, l2);
    h1 = fma(w, ex * ex + ey * ey, h1);
    en = fma(w * a, (K[0] * ex + K[1] * ey) * ex + (K[2] * ex + K[3] * ey) * ey, en);
  }
  out[k] = l2;
  out[size_t(m.n_own) + k] = h1;
  out[2 * size_t(m.n_own) + k] = en;
}

// Lagrange nodes of Elem<KIND, P> in reference coordinates, in DoF order (device.cuh)
template <int KIND, int P>
__device__ __forceinline__ void reference_node(int i, double& xi, double& eta) {
  if constexpr (KIND == HDD_SIMPLEX2D && P == 1) {
    xi = i == 1 ? 1.0 : 0.0;
    eta = i == 2 ? 1.0 : 0.0;
  } else if constexpr (KIND == HDD_SIMPLEX2D) {  // (0,0) (1/2,0) (1,0) (0,1/2) (1/2,1/2) (0,1)
    const int row = i < 3 ? 0 : i < 5 ? 1 : 2, in_row = i < 3 ? i : i < 5 ? i - 3 : 0;
    xi = 0.5 * in_row;
    eta = 0.5 * row;
  } else {  // tensor product, x fastest
    xi = double(i % (P + 1)) / P;
    eta = double(i / (P + 1)) / P;
  }
}

// GDT::Operators::Prolongation (test/linearelliptic.hh:168-176): every DoF of the fine DG function is the value of the
// coarse DG function at the fine Lagrange node, the coarse function being the polynomial of the father cell (the coarse
// cell that contains the fine cell; hdd_grid_fathers).  One thread per fine cell, no neighbour access: a fine cell
// inherits from its father only, like the reference's local L2 projection of a function that is polynomial on the cell.
template <int KIND, int PC, int PF>
__global__ void __launch_bounds__(128)
    k_prolong(MeshView fine, const double* __restrict__ cgeo_coarse, int32_t n_coarse, const int32_t* __restrict__ father,
              const double* __restrict__ u_coarse, double* __restrict__ u_fine, int* __restrict__ flag) {
  using GC = Elem<KIND, PC>;
  using GF = Elem<KIND, PF>;
  constexpr int NC = GC::NL, NFINE = GF::NL;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= fine.n_own) return;
  const int fa = __ldg(father + k);
  if (fa < 0 || fa >= n_coarse) {
    atomicOr(flag, 1);
    return;
  }
  GF gf;
  gf.load(fine.cgeo, fine.own0 + k);
  GC gc;
  gc.load(cgeo_coarse, fa);
  double u[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) u[j] = __ldg(u_coarse + size_t(NC) * fa + j);
#pragma unroll
  for (int i = 0; i < NFINE; ++i) {
    double xi, eta, x, y, a, b, phi[NC], gx[NC], gy[NC];
    reference_node<KIND, PF>(i, xi, eta);
    gf.to_global(xi, eta, x, y);
    gc.to_local(x, y, a, b);
    gc.basis(a, b, phi, gx, gy);
    double v = 0.0;
#pragma unroll
    for (int j = 0; j < NC; ++j) v = fma(u[j], phi[j], v);
    u_fine[size_t(NFINE) * k + i] = v;
  }
}

// per-segment partial dot products (deterministic: fixed tree inside the block, host adds the segments in order)
__global__ void __launch_bounds__(256)
    k_segment_dot(const double* __restrict__ x, const double* __restrict__ y, const int64_t* __restrict__ seg, int nd,
                  double* __restrict__ out) {
  __shared__ double sm[256];
  const int64_t b = seg[blockIdx.x] * nd, e = seg[blockIdx.x + 1] * nd;
  double v = 0.0;
  for (int64_t i = b + threadIdx.x; i < e; i += blockDim.x) v = fma(x[i], y[i], v);
  sm[threadIdx.x] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (int(threadIdx.x) < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sm[0];
}

}  // namespace

void launch_fill_volume_csr(const MeshView& m, int64_t* rowptr, int32_t* col, cudaStream_t s) {
  const int64_t rows = int64_t(m.n_own) * m.nl;
  dispatch_nl(m.nl, [&](auto nl) {
    k_fill_volume_csr<decltype(nl)::value><<<int((rows + 1 + 255) / 256), 256, 0, s>>>(m, rowptr, col);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_block_spmv(const MeshView& m, const double* values, const double* x_own, double* y, cudaStream_t s) {
  const int64_t rows = int64_t(m.n_own) * m.nl;
  if (rows == 0) return;
  const int blocks = int(std::min<int64_t>((rows + kThreads - 1) / kThreads, 148 * 8));
  dispatch_nl(m.nl, [&](auto nl) { k_block_spmv<decltype(nl)::value><<<blocks, kThreads, 0, s>>>(rows, values, x_own, y); });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_error_norms(const MeshView& m, int polorder, const DevFn& exact, const DevFn& exact_dx, const DevFn& exact_dy,
                        const DevCombo& factor, const DevFn* fn_table, int order, const double* u_own, double* out,
                        cudaStream_t s) {
  if (m.n_own == 0) return;
  const ElemRule rule = element_rule(m.kind, order);
  const int blocks = (m.n_own + 127) / 128;
  auto go = [&](auto kind, auto p) {
    k_error_norms<decltype(kind)::value, decltype(p)::value>
        <<<blocks, 128, 0, s>>>(m, exact, exact_dx, exact_dy, factor, fn_table, rule, u_own, out);
  };
  if (m.kind == HDD_SIMPLEX2D) {
    if (polorder == 1) go(ic<HDD_SIMPLEX2D>{}, ic<1>{}); else go(ic<HDD_SIMPLEX2D>{}, ic<2>{});
  } else {
    if (polorder == 1) go(ic<HDD_CUBE2D>{}, ic<1>{}); else go(ic<HDD_CUBE2D>{}, ic<2>{});
  }
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_prolong(const MeshView& fine, int p_fine, const double* cgeo_coarse, int32_t n_coarse, int p_coarse,
                    const int32_t* father, const double* u_coarse, double* u_fine, int* flag, cudaStream_t s) {
  if (fine.n_own == 0) return;
  const int blocks = (fine.n_own + 127) / 128;
  auto go = [&](auto kind, auto pc, auto pf) {
    k_prolong<decltype(kind)::value, decltype(pc)::value, decltype(pf)::value>
        <<<blocks, 128, 0, s>>>(fine, cgeo_coarse, n_coarse, father, u_coarse, u_fine, flag);
  };
  auto by_p = [&](auto kind) {
    if (p_coarse == 1 && p_fine == 1) go(kind, ic<1>{}, ic<1>{});
    else if (p_coarse == 1) go(kind, ic<1>{}, ic<2>{});
    else if (p_fine == 1) go(kind, ic<2>{}, ic<1>{});
    else go(kind, ic<2>{}, ic<2>{});
  };
  if (fine.kind == HDD_SIMPLEX2D) by_p(ic<HDD_SIMPLEX2D>{}); else by_p(ic<HDD_CUBE2D>{});
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_segment_dot(const double* x, const double* y, const int64_t* seg_ptr_dev, int n_seg, int nd, double* out,
                        cudaStream_t s) {
  if (n_seg == 0) return;
  k_segment_dot<<<n_seg, 256, 0, s>>>(x, y, seg_ptr_dev, nd, out);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

}  // namespace hdd
