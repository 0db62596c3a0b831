// K7-K10: ESV2007 / OS2014 local indicators on 2-d simplices for sm_100a.
//
// Two passes instead of the reference's four grid walks (estimators/swipdg.hh:668-687):
//   pass 1 (per vertex)  Oswald value = mean of the DG values around the vertex, 0 on the boundary
//                        (GDT::Operators::OswaldInterpolation, estimators/swipdg.hh:149-150)
//   pass 2 (per cell)    everything else, one thread per element.  The RT0 flux reconstruction
//                        (Operators::DiffusiveFluxReconstruction, estimators/swipdg.hh:590-595) is evaluated
//                        owner-computes: each cell integrates the SWIPDG flux through its own three faces with its
//                        own outward normal - the flux is antisymmetric under swapping the two cells, so no face
//                        array and no face pass are needed - and immediately consumes t_h in eta_DF, eta_DF*, eta_R*.
#include "kernels.hpp"

namespace hdd {

namespace {

__global__ void k_vertex_means(const int64_t* __restrict__ vptr, const int32_t* __restrict__ vdof,
                               const uint8_t* __restrict__ vboundary, int32_t n_verts, const double* __restrict__ u,
                               double* __restrict__ vm) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_verts) return;
  if (vboundary[v]) { vm[v] = 0.0; return; }
  const int64_t b = vptr[v], e = vptr[v + 1];
  double s = 0.0;
  for (int64_t k = b; k < e; ++k) s += u[vdof[k]];
  vm[v] = e > b ? s / double(e - b) : 0.0;
}

constexpr double kPi = 3.14159265358979323846264338327950288;

// The quadrature tables of one estimator pass (6.4 KB).  They travel as a __grid_constant__ kernel parameter: every
// lane reads the same entry at the same time, which the constant bank serves as a broadcast - no global-memory table,
// no allocation and no synchronisation around the launch.
struct IndicatorRules {
  ElemRule nc, p0, res, df, cut, amin, amax;
  LineRule face;
};

// sum_k theta_k f_k for a combination whose members are all constants or per-cell values
__device__ __forceinline__ double combo_cell(const DevCombo& c, const DevFn* table, int cell) {
  double s = 0.0;
  for (int k = 0; k < c.n; ++k) {
    const DevFn& f = table[c.idx[k]];
    s += c.theta[k] * (f.kind == HDD_FN_CONSTANT ? f.value : __ldg(f.cell + cell));
  }
  return s;
}

// One thread per element, everything in registers: no per-thread array is indexed dynamically (geometry, DoFs and
// fluxes are addressed with compile-time indices, the expression interpreter runs on a register stack), so nothing
// spills to local memory.  EXPR = false: every diffusion-factor combination is constant per cell (Constant / per-cell
// data: ESV2007, SPE10) and is evaluated once per cell instead of once per quadrature point.
// The P1 functions are evaluated as u(x) = u_0 + grad u . (x - v_0) instead of through the basis at mapped-back points.
// TRIG: the force is c cos(..) cos(..) of affine arguments (TrigProduct, expr.hpp; the ESV2007 force) and travels as plain
// scalars: per cell the arguments become affine in the reference coordinates, per point the force is two fused
// multiply-adds and one branch-free fast_cos per factor - straight-line code the compiler interleaves over the unrolled
// points, instead of the table-driven FastFn loop around the library cos() (ncu, round 2: 8900 instructions per cell, 29 %
// of them fp64, half of the stall samples waiting on fixed-latency dependencies).
template <bool EXPR, bool TRIG>
__global__ void __launch_bounds__(128, 4)
    k_indicators(const __grid_constant__ MeshView m, const __grid_constant__ IndicatorArgs a,
                 const __grid_constant__ IndicatorRules R, const __grid_constant__ TrigProduct tp, double s_in, double s_bnd) {
  using G = Geo<HDD_SIMPLEX2D>;
  constexpr int NL = 3;
  // the data functions (expression programs included) are staged in shared memory once per block
  extern __shared__ __align__(16) unsigned char fn_smem[];
  DevFn* table = reinterpret_cast<DevFn*>(fn_smem);
  {
    const int words = a.n_fn * int(sizeof(DevFn) / 4);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.fn_table);
    uint32_t* dst = reinterpret_cast<uint32_t*>(fn_smem);
    for (int w = threadIdx.x; w < words; w += blockDim.x) dst[w] = src[w];
  }
  __syncthreads();
  const DevFn& force = table[a.force_idx];
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  const int c = m.own0 + k;
  G g;
  g.load(m.cgeo, c);
  double K[4];
  load_tensor(m.tensor, c, K);
  const double tr = K[0] + K[3], det = K[0] * K[3] - K[1] * K[2];
  const double lam_min = 0.5 * tr - sqrt(fmax(0.0, 0.25 * tr * tr - det));
  // physical gradients of the barycentric coordinates (constant on the cell)
  const double g1x = g.i00, g1y = g.i01, g2x = g.i10, g2y = g.i11, g0x = -g.i00 - g.i10, g0y = -g.i01 - g.i11;
  const double u0 = a.u_local[size_t(NL) * c], u1 = a.u_local[size_t(NL) * c + 1], u2 = a.u_local[size_t(NL) * c + 2];
  const double ux = u0 * g0x + u1 * g1x + u2 * g2x, uy = u0 * g0y + u1 * g1y + u2 * g2y;
  double dx, dy;
  {
    const double d0 = u0 - a.vertex_mean[a.cell_verts[size_t(NL) * k]];
    const double d1 = u1 - a.vertex_mean[a.cell_verts[size_t(NL) * k + 1]];
    const double d2 = u2 - a.vertex_mean[a.cell_verts[size_t(NL) * k + 2]];
    dx = d0 * g0x + d1 * g1x + d2 * g2x;
    dy = d0 * g0y + d1 * g1y + d2 * g2y;
  }
  // per-cell factor values (EXPR = false)
  double c_mu = 0.0, c_hat = 0.0;
  if (!EXPR) {
    c_mu = combo_cell(a.a_mu, table, c);
    c_hat = combo_cell(a.a_hat, table, c);
  }
  const size_t n = size_t(m.n_own);
  // eta_NC,T^2 = int_T a(mu_bar) K grad(u - Iu) . grad(u - Iu)
  double v_nc;
  {
    const double e = (K[0] * dx + K[1] * dy) * dx + (K[2] * dx + K[3] * dy) * dy;
    double s = 0.0;
    if (EXPR) {
      for (int q = 0; q < R.nc.n; ++q) {
        double x, y;
        g.to_global(R.nc.x[q], R.nc.y[q], x, y);
        s += R.nc.w[q] * g.detj * combo_eval(a.a_bar, table, c, x, y) * e;
      }
    } else {
      const double ab = combo_cell(a.a_bar, table, c);
      for (int q = 0; q < R.nc.n; ++q) s += R.nc.w[q] * g.detj * ab * e;
    }
    a.out[0 * n + k] = s;
    v_nc = s;
  }
  // c_T of the Cutoff weight and the OS2014 minimum over the parameter range
  double cT = 1e300;
  if (EXPR) {
    for (int q = 0; q < R.cut.n; ++q) {
      double x, y;
      g.to_global(R.cut.x[q], R.cut.y[q], x, y);
      cT = fmin(cT, combo_eval(a.a_cut, table, c, x, y) * lam_min);
    }
  } else {
    cT = combo_cell(a.a_cut, table, c) * lam_min;
  }
  const double hT = g.diameter();
  const double cutoff = hT * hT / (kPi * kPi * cT);
  {
    double mn = 1e300;
    if (EXPR) {
      for (int q = 0; q < R.amin.n; ++q) {
        double x, y;
        g.to_global(R.amin.x[q], R.amin.y[q], x, y);
        mn = fmin(mn, combo_eval(a.a_min, table, c, x, y));
      }
      for (int q = 0; q < R.amax.n; ++q) {
        double x, y;
        g.to_global(R.amax.x[q], R.amax.y[q], x, y);
        mn = fmin(mn, combo_eval(a.a_max, table, c, x, y));
      }
    } else {
      mn = fmin(combo_cell(a.a_min, table, c), combo_cell(a.a_max, table, c));
    }
    a.out[6 * n + k] = mn * lam_min;
  }
  // outward RT0 fluxes G_f = int_f ( -{{A grad u . n}}_omega + pen [[u]] )  resp. ( -A grad u . n + pen u ); the three
  // faces are written out with compile-time vertex indices: {0,1}, {0,2}, {1,2}
  const double kux = K[0] * ux + K[1] * uy, kuy = K[2] * ux + K[3] * uy;
  double cx, cy;
  g.centroid(cx, cy);
  auto face_flux = [&](const double ax, const double ay, const double bx, const double by, const int nbc) -> double {
    const double tx = bx - ax, ty = by - ay;
    const double h = sqrt(tx * tx + ty * ty), ih = 1.0 / h;
    double nx = ty * ih, ny = -tx * ih;
    if (nx * (0.5 * (ax + bx) - cx) + ny * (0.5 * (ay + by) - cy) < 0.0) { nx = -nx; ny = -ny; }
    const double dm = nx * (K[0] * nx + K[1] * ny) + ny * (K[2] * nx + K[3] * ny);
    const double fm1 = kux * nx + kuy * ny;  // K grad u . n
    double s = 0.0;
    if (nbc < 0) {
      for (int q = 0; q < R.face.n; ++q) {
        const double x = ax + R.face.x[q] * tx, y = ay + R.face.x[q] * ty;
        const double uv = u0 + ux * (x - g.vx[0]) + uy * (y - g.vy[0]);
        const double am = EXPR ? combo_eval(a.a_mu, table, c, x, y) : c_mu;
        s += R.face.w[q] * h * (-am * fm1 + s_bnd * dm * am * ih * uv);
      }
    } else {
      G gn;
      gn.load(m.cgeo, nbc);
      double Kn[4];
      load_tensor(m.tensor, nbc, Kn);
      const double n0 = a.u_local[size_t(NL) * nbc], n1 = a.u_local[size_t(NL) * nbc + 1], n2 = a.u_local[size_t(NL) * nbc + 2];
      const double vx = n0 * (-gn.i00 - gn.i10) + n1 * gn.i00 + n2 * gn.i10;
      const double vy = n0 * (-gn.i01 - gn.i11) + n1 * gn.i01 + n2 * gn.i11;
      const double dp = nx * (Kn[0] * nx + Kn[1] * ny) + ny * (Kn[2] * nx + Kn[3] * ny);
      const double gamma = dp * dm / (dp + dm), wm = dp / (dp + dm), wp = dm / (dp + dm);
      const double fp1 = (Kn[0] * vx + Kn[1] * vy) * nx + (Kn[2] * vx + Kn[3] * vy) * ny;
      const double c_ne = EXPR ? 0.0 : combo_cell(a.a_mu, table, nbc);
      for (int q = 0; q < R.face.n; ++q) {
        const double x = ax + R.face.x[q] * tx, y = ay + R.face.x[q] * ty;
        const double um = u0 + ux * (x - g.vx[0]) + uy * (y - g.vy[0]);
        const double up = n0 + vx * (x - gn.vx[0]) + vy * (y - gn.vy[0]);
        const double am = EXPR ? combo_eval(a.a_mu, table, c, x, y) : c_mu;
        const double ap = EXPR ? combo_eval(a.a_mu, table, nbc, x, y) : c_ne;
        const double pen = s_in * gamma * 0.5 * (am + ap) * ih;
        s += R.face.w[q] * h * (-(wm * am * fm1 + wp * ap * fp1) + pen * (um - up));
      }
    }
    return s;
  };
  const double G0 = face_flux(g.vx[0], g.vy[0], g.vx[1], g.vy[1], m.neigh[size_t(3) * k]);
  const double G1 = face_flux(g.vx[0], g.vy[0], g.vx[2], g.vy[2], m.neigh[size_t(3) * k + 1]);
  const double G2 = face_flux(g.vx[1], g.vy[1], g.vx[2], g.vy[2], m.neigh[size_t(3) * k + 2]);
  const double area = 0.5 * g.detj;
  const double div = (G0 + G1 + G2) / area;
  // P0 projection of f, then int_T (f - P0 f)^2 and int_T (f - div t_h)^2 in one sweep over the residual rule: the force
  // (the expensive part: an interpreted expression per point) is evaluated once per point and never stored
  // TRIG: theta_k(xi, eta) = t0_k + tx_k xi + ty_k eta, the affine argument of factor k in the reference coordinates
  double t00 = 0.0, t0x = 0.0, t0y = 0.0, t10 = 0.0, t1x = 0.0, t1y = 0.0;
  bool trig = false;
  if (TRIG) {
    const double e1x = g.vx[1] - g.vx[0], e1y = g.vy[1] - g.vy[0], e2x = g.vx[2] - g.vx[0], e2y = g.vy[2] - g.vy[0];
    t00 = fma(tp.a[0], g.vx[0], fma(tp.b[0], g.vy[0], tp.d[0]));
    t0x = tp.a[0] * e1x + tp.b[0] * e1y;
    t0y = tp.a[0] * e2x + tp.b[0] * e2y;
    t10 = fma(tp.a[1], g.vx[0], fma(tp.b[1], g.vy[0], tp.d[1]));
    t1x = tp.a[1] * e1x + tp.b[1] * e1y;
    t1y = tp.a[1] * e2x + tp.b[1] * e2y;
    // the whole cell inside the range of fast_cos (always, for any sensible domain); otherwise the general evaluation
    trig = fabs(t00) + fabs(t0x) + fabs(t0y) < kFastCosMax && fabs(t10) + fabs(t1x) + fabs(t1y) < kFastCosMax;
  }
  auto force_at = [&](const double xi, const double eta) -> double {
    return tp.c * fast_cos(fma(t0x, xi, fma(t0y, eta, t00))) * fast_cos(fma(t1x, xi, fma(t1y, eta, t10)));
  };
  double f0 = 0.0;
  if (TRIG && trig) {
#pragma unroll 7
    for (int q = 0; q < R.p0.n; ++q) f0 = fma(R.p0.w[q], force_at(R.p0.x[q], R.p0.y[q]), f0);
  } else {
#pragma unroll 4
    for (int q = 0; q < R.p0.n; ++q) {
      double x, y;
      g.to_global(R.p0.x[q], R.p0.y[q], x, y);
      f0 += R.p0.w[q] * fn_eval(force, c, x, y);
    }
  }
  f0 /= 0.5;
  double v_r;
  {
    double rs = 0.0, rstar = 0.0;
    if (TRIG && trig) {
#pragma unroll 5
      for (int q = 0; q < R.res.n; ++q) {
        const double fv = force_at(R.res.x[q], R.res.y[q]);
        const double d = fv - f0, ds = fv - div;
        const double w = R.res.w[q] * g.detj;
        rs = fma(w * d, d, rs);
        rstar = fma(w * ds, ds, rstar);
      }
    } else {
#pragma unroll 4
      for (int q = 0; q < R.res.n; ++q) {
        double x, y;
        g.to_global(R.res.x[q], R.res.y[q], x, y);
        const double fv = fn_eval(force, c, x, y);
        const double d = fv - f0, ds = fv - div;
        rs += R.res.w[q] * g.detj * d * d;
        rstar += R.res.w[q] * g.detj * ds * ds;
      }
    }
    a.out[1 * n + k] = rs;
    a.out[2 * n + k] = cutoff * rs;
    a.out[5 * n + k] = cutoff * rstar;
    a.out[7 * n + k] = rstar;
    v_r = cutoff * rs;
  }
  // eta_DF, eta_DF*: t_h(x) = sum_f G_f (x - p_f) / (2 |T|), p_f the vertex opposite face f: {0,1}->2, {0,2}->1, {1,2}->0
  double v_df;
  {
    double s = 0.0, ss = 0.0;
    const double k00 = K[3] / det, k01 = -K[1] / det, k10 = -K[2] / det, k11 = K[0] / det;
    for (int q = 0; q < R.df.n; ++q) {
      double x, y;
      g.to_global(R.df.x[q], R.df.y[q], x, y);
      const double t0 = (G0 * (x - g.vx[2]) + G1 * (x - g.vx[1]) + G2 * (x - g.vx[0])) / (2.0 * area);
      const double t1 = (G0 * (y - g.vy[2]) + G1 * (y - g.vy[1]) + G2 * (y - g.vy[0])) / (2.0 * area);
      const double ah = EXPR ? combo_eval(a.a_hat, table, c, x, y) : c_hat;
      const double am = EXPR ? combo_eval(a.a_mu, table, c, x, y) : c_mu;
      const double w = R.df.w[q] * g.detj;
      double v0 = ah * kux + t0, v1 = ah * kuy + t1;
      s += w * (v0 * (k00 * v0 + k01 * v1) + v1 * (k10 * v0 + k11 * v1)) / ah;
      v0 = am * kux + t0;
      v1 = am * kuy + t1;
      ss += w * (v0 * (k00 * v0 + k01 * v1) + v1 * (k10 * v0 + k11 * v1)) / ah;
    }
    a.out[3 * n + k] = s;
    a.out[4 * n + k] = ss;
    v_df = s;
  }
  // eta_T^2 of eta_ESV2007 (estimators/swipdg.hh:683-684)
  const double t = sqrt(v_r) + sqrt(v_df);
  a.out[8 * n + k] = v_nc + t * t;
}

// Deterministic segmented reduction of `n_rows` rows in one launch (row r of `in` starts at r * row_stride): one block
// per (segment, row), fixed tree.  The mesh cuts the owned cells of every subdomain into segments of at most 8192 cells
// (mesh.cu), so the grid is n_own / 8192 x n_rows blocks; the host adds the segment results per subdomain in order.
// Rows whose bit is set in min_mask are reduced with min instead of +.
__global__ void __launch_bounds__(256)
    k_segment_reduce(const double* __restrict__ in, int64_t row_stride, unsigned min_mask, const int64_t* __restrict__ seg,
                     double* __restrict__ out) {
  __shared__ double sm[256];
  const int sg = blockIdx.x, row = blockIdx.y, n_seg = gridDim.x;
  const bool is_min = (min_mask >> row) & 1u;
  const int64_t b = seg[sg], e = seg[sg + 1];
  const double* src = in + int64_t(row) * row_stride;
  double v = is_min ? 1e300 : 0.0;
  for (int64_t i = b + threadIdx.x; i < e; i += 256) v = is_min ? fmin(v, src[i]) : v + src[i];
  sm[threadIdx.x] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (int(threadIdx.x) < o) sm[threadIdx.x] = is_min ? fmin(sm[threadIdx.x], sm[threadIdx.x + o]) : sm[threadIdx.x] + sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[size_t(row) * n_seg + sg] = sm[0];
}

}  // namespace

void launch_oswald_vertex_means(const int64_t* vptr, const int32_t* vdof, const uint8_t* vboundary, int32_t n_verts,
                                const double* u_local, double* vertex_mean, cudaStream_t s) {
  if (n_verts == 0) return;
  k_vertex_means<<<(n_verts + 255) / 256, 256, 0, s>>>(vptr, vdof, vboundary, n_verts, u_local, vertex_mean);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

static bool combo_is_cellwise(const DevCombo& c, const DevFn* host_table) {
  for (int k = 0; k < c.n; ++k)
    if (host_table[c.idx[k]].kind == HDD_FN_EXPRESSION) return false;
  return true;
}

void launch_indicators(const MeshView& m, const IndicatorArgs& a, const DevFn* fn_table_host, int polorder, cudaStream_t s) {
  if (m.n_own == 0) return;
  if (m.kind != HDD_SIMPLEX2D)
    HDD_THROW(HDD_ERR_USING_THIS_WRONG, "estimators are only available on 2d simplex grids (estimators/swipdg.hh:71)");
  const int p = polorder, over = 2;  // over_integrate, estimators/swipdg.hh:47
  IndicatorRules R;
  R.nc = triangle_rule(a.a_bar.order + 2 * (p - 1) + over);
  R.p0 = triangle_rule(a.force_order + over);
  R.res = triangle_rule(2 * a.force_order + over);
  R.df = triangle_rule(a.a_hat.order + 2 * p + over);
  R.cut = triangle_rule(a.a_cut.order + over);
  R.amin = triangle_rule(a.a_min.order);
  R.amax = triangle_rule(a.a_max.order);
  R.face = line_rule(a.a_mu.order + 2 * p + over);
  static_assert(sizeof(DevFn) % 4 == 0, "DevFn must be word sized");
  const size_t fn_bytes = size_t(a.n_fn) * sizeof(DevFn);
  if (fn_bytes > 48 * 1024) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "too many data functions for the estimator kernel");
  const bool expr = !(combo_is_cellwise(a.a_mu, fn_table_host) && combo_is_cellwise(a.a_hat, fn_table_host) &&
                      combo_is_cellwise(a.a_bar, fn_table_host) && combo_is_cellwise(a.a_cut, fn_table_host) &&
                      combo_is_cellwise(a.a_min, fn_table_host) && combo_is_cellwise(a.a_max, fn_table_host));
  const int grid = (m.n_own + 127) / 128;
  const DevFn& force = fn_table_host[a.force_idx];
  TrigProduct tp{};
  if (force.kind == HDD_FN_EXPRESSION && force.fast.n_terms > 0) tp = as_trig_product(force.fast);
  const double si = sigma_inner(p), sb = sigma_boundary(p);
  if (expr && tp.valid)
    k_indicators<true, true><<<grid, 128, fn_bytes, s>>>(m, a, R, tp, si, sb);
  else if (expr)
    k_indicators<true, false><<<grid, 128, fn_bytes, s>>>(m, a, R, tp, si, sb);
  else if (tp.valid)
    k_indicators<false, true><<<grid, 128, fn_bytes, s>>>(m, a, R, tp, si, sb);
  else
    k_indicators<false, false><<<grid, 128, fn_bytes, s>>>(m, a, R, tp, si, sb);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_segment_reduce(const double* in, int64_t row_stride, int n_rows, unsigned min_mask, const int64_t* seg_ptr_dev,
                           int n_seg, double* out, cudaStream_t s) {
  if (n_seg == 0 || n_rows == 0) return;
  k_segment_reduce<<<dim3(unsigned(n_seg), unsigned(n_rows)), 256, 0, s>>>(in, row_stride, min_mask, seg_ptr_dev, out);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_segment_sums(const double* in, const int64_t* seg_ptr_dev, int n_seg, double* out, cudaStream_t s) {
  launch_segment_reduce(in, 0, 1, 0u, seg_ptr_dev, n_seg, out, s);
}

void launch_segment_min(const double* in, const int64_t* seg_ptr_dev, int n_seg, double* out, cudaStream_t s) {
  launch_segment_reduce(in, 0, 1, 1u, seg_ptr_dev, n_seg, out, s);
}

}  // namespace hdd
