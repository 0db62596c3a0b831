// K5 (SpMV) and K6 (fused CG vector updates) for sm_100a.
//
// Matrix storage: the CSR value array of the owned rows (bit-compatible with what hdd_component_values hands out),
// but the kernels never read CSR column indices or row pointers.  The DG matrix is block structured - every row of
// cell T has one dense n_loc-wide run per member of sort({T} u neighbours) - so the column structure is recovered
// from the 16-byte neighbour record of the cell and one 8-byte block offset per cell.  That removes the 4 B/nnz
// index stream of textbook CSR: 8.05 B/nnz instead of 12 B/nnz of HBM traffic for Q1.
//
// Two SpMV kernels:
//   k_cg_spmv      generic (P1 and Q1): one thread per row, 256-bit loads for Q1.
//   k_cg_spmv_tma  Q1: the matrix stream (88 % of the bytes) is moved by the TMA engine.  The row blocks of
//                  consecutive cells are one contiguous byte range, so a producer warp issues 1-D bulk copies
//                  (cp.async.bulk, UBLKCP) of 8-cell tiles into a 32-stage shared-memory ring guarded by mbarriers;
//                  16 consumer warps read their rows from shared memory, gather x through L1/L2 and write q.
//                  The copy engine keeps ~160 KB per SM in flight independent of what the consumer warps wait on.
//
// CG is the classic Hestenes-Stiefel recurrence (same algebra as oracle/or_cg) with device-resident scalars:
// no host synchronisation inside the iteration, dot products reduced deterministically (fixed per-block partials,
// last-arriving block sums them in a fixed order), convergence latched in a ping-pong flag so that iterations
// launched after convergence are no-ops.  Preconditioners: identity, diagonal (Jacobi), and the cell-block diagonal
// (block Jacobi with the n_loc x n_loc diagonal blocks, the natural choice for DG).
#include <cstdlib>

#include "kernels.hpp"
#include "reduce.cuh"

namespace hdd {

namespace {

constexpr int kCgThreads = 256;

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

// cells of the row block of owned cell k in ascending (= column) order; returns the number of blocks
template <int NF>
__device__ __forceinline__ int sorted_blocks(const MeshView& m, int k, int* cells) {
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  const int self = m.own0 + k;
  int nblk = 1;
#pragma unroll
  for (int f = 0; f < NF; ++f) nblk += nb[f] >= 0 ? 1 : 0;
#pragma unroll
  for (int s = 0; s < NF + 1; ++s) cells[s] = 0;
  {
    const int slot = block_slot<NF>(self, nb, self);
#pragma unroll
    for (int s = 0; s < NF + 1; ++s)
      if (s == slot) cells[s] = self;
  }
#pragma unroll
  for (int f = 0; f < NF; ++f)
    if (nb[f] >= 0) {
      const int slot = block_slot<NF>(self, nb, nb[f]);
#pragma unroll
      for (int s = 0; s < NF + 1; ++s)
        if (s == slot) cells[s] = nb[f];
    }
  return nblk;
}

__device__ __forceinline__ void ld256_stream(const double* p, double& a, double& b, double& c, double& d) {
  asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void ld256(const double* p, double& a, double& b, double& c, double& d) {
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
// read-modify-write streams (x, r, p) must not use the non-coherent path
__device__ __forceinline__ void ld256_rw(const double* p, double& a, double& b, double& c, double& d) {
  asm volatile("ld.global.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ void st256(double* p, double a, double b, double c, double d) {
  asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

__device__ __forceinline__ double* dir_in(const CgBuffers& c, int par) { return (c.p_alt && par) ? c.p_alt : c.p; }
__device__ __forceinline__ double* dir_out(const CgBuffers& c, int par) {
  return c.p_alt ? (par ? c.p : c.p_alt) : c.p;  // ping-pong: iteration `par` writes the other buffer
}

// Row kernel shared by SpMV and the CG step: y_t = sum over the blocks of row t, ascending column order.
template <int NF, int NL>
__device__ __forceinline__ double row_times_x(const MeshView& m, const double* __restrict__ vals,
                                              const double* __restrict__ x, int64_t t) {
  const int k = int(t / NL), i = int(t % NL);
  int cells[NF + 1];
  const int nblk = sorted_blocks<NF>(m, k, cells);
  const double* row = vals + m.blk_start[k] * (NL * NL) + int64_t(i) * nblk * NL;
  double sum = 0.0;
#pragma unroll
  for (int s = 0; s < NF + 1; ++s) {
    if (s < nblk) {
      const double* xs = x + size_t(NL) * cells[s];
      if constexpr (NL == 4) {
        double a0, a1, a2, a3, x0, x1, x2, x3;
        ld256_stream(row + s * 4, a0, a1, a2, a3);
        ld256(xs, x0, x1, x2, x3);
        sum = fma(a0, x0, sum); sum = fma(a1, x1, sum); sum = fma(a2, x2, sum); sum = fma(a3, x3, sum);
      } else {
#pragma unroll
        for (int j = 0; j < NL; ++j) sum = fma(__ldg(row + s * NL + j), __ldg(xs + j), sum);
      }
    }
  }
  return sum;
}

template <int NF, int NL>
__global__ void __launch_bounds__(kCgThreads)
    k_spmv(MeshView m, const double* __restrict__ vals, const double* __restrict__ x, double* __restrict__ y) {
  const int64_t rows = int64_t(m.n_own) * NL;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < rows; t += stride)
    y[t] = row_times_x<NF, NL>(m, vals, x, t);
}

template <int NF, int NL>
__global__ void __launch_bounds__(kCgThreads) k_cg_spmv(MeshView m, CgBuffers c, int par) {
  CgScalars* sc = c.sc;
  if (sc->done[par]) return;
  const int64_t rows = int64_t(m.n_own) * NL, own_off = int64_t(m.own0) * NL;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  double v[1] = {0.0};
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < rows; t += stride) {
    const double* pc = dir_in(c, par);
    const double y = row_times_x<NF, NL>(m, c.values, pc, t);
    c.q[t] = y;
    v[0] = fma(pc[own_off + t], y, v[0]);
  }
  grid_sum<1>(v, c.partial, &sc->ticket_a, [sc](const double(&w)[1]) { sc->red[0] = w[0]; });
}

// ---- TMA-staged Q1 SpMV -----------------------------------------------------------------------------------------
constexpr int kTmaStages = 32;
constexpr int kTmaTileCells = 8;                           // one warp: 8 cells x 4 rows
constexpr int kTmaStageBytes = kTmaTileCells * 5 * 128;    // 8 cells x <= 5 blocks x 16 doubles
constexpr int kTmaConsumerWarps = 16;
constexpr int kTmaThreads = (kTmaConsumerWarps + 1) * 32;
constexpr int kTmaSmemBytes = kTmaStages * kTmaStageBytes + 2 * kTmaStages * 8;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// direction entries of one cell: owned cells come from this rank's buffer; in peer-memory mode halo cells are formed on
// the fly from the owner's residual and previous direction, read through NVLink (p = D^-1 r + beta p_old)
__device__ __forceinline__ void load_direction(const double* p_cur, const PeerView& pv, int par, double beta, bool first,
                                               int cell, double* v) {
  if (!pv.enabled || (cell >= pv.own0 && cell < pv.own0 + pv.n_own)) {
    ld256(p_cur + size_t(4) * cell, v[0], v[1], v[2], v[3]);
    return;
  }
  const int h = cell < pv.own0 ? cell : cell - pv.n_own;
  const int peer = __ldg(pv.halo_peer + h), rc = __ldg(pv.halo_rcell + h);
  double r[4], d[4];
  ld256_rw(pv.r[peer] + size_t(4) * rc, r[0], r[1], r[2], r[3]);
  ld256(pv.dinv_local + size_t(4) * cell, d[0], d[1], d[2], d[3]);
#pragma unroll
  for (int j = 0; j < 4; ++j) v[j] = d[j] * r[j];
  if (!first) {
    double po[4];
    ld256_rw(pv.p[par ^ 1][peer] + size_t(4) * (pv.own0_of[peer] + rc), po[0], po[1], po[2], po[3]);
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = fma(beta, po[j], v[j]);
  }
}

__global__ void __launch_bounds__(kTmaThreads, 1)
    k_cg_spmv_tma(MeshView m, CgBuffers c, int par, int cells_per_cta, const __grid_constant__ PeerView pv) {
  constexpr int NL = 4, NF = 4;
  extern __shared__ __align__(128) unsigned char smem[];
  CgScalars* sc = c.sc;
  if (sc->done[par]) return;
  unsigned char* stage_base = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kTmaStages * kTmaStageBytes);
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + kTmaStages);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kTmaStages; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int c0 = blockIdx.x * cells_per_cta;
  const int c1 = min(c0 + cells_per_cta, m.n_own);
  const int n_tiles = c1 > c0 ? (c1 - c0 + kTmaTileCells - 1) / kTmaTileCells : 0;
  double v[1] = {0.0};
  if (warp == kTmaConsumerWarps) {
    // producer: lane l owns stage l and feeds tiles l, l+32, ...
    for (int t = lane; t < n_tiles; t += kTmaStages) {
      const int n = t / kTmaStages;
      if (n > 0) mbar_wait(empty0 + 8 * lane, (n - 1) & 1);
      const int k0 = c0 + t * kTmaTileCells, k1 = min(k0 + kTmaTileCells, c1);
      const int64_t b0 = __ldg(m.blk_start + k0), b1 = __ldg(m.blk_start + k1);
      const uint32_t bytes = uint32_t(b1 - b0) * (NL * NL * 8);
      mbar_expect_tx(full0 + 8 * lane, bytes);
      bulk_g2s(smem_u32(stage_base + lane * kTmaStageBytes), c.values + b0 * (NL * NL), bytes, full0 + 8 * lane);
    }
  } else {
    const int64_t own_off = int64_t(m.own0) * NL;
    const int i = lane & 3;
    const double* p_cur = dir_in(c, par);
    const bool first = sc->it[par] == 0;
    const double beta = (pv.enabled && !first) ? sc->rz[par] / sc->rz[par ^ 1] : 0.0;
    for (int t = warp; t < n_tiles; t += kTmaConsumerWarps) {
      const int stage = t % kTmaStages, n = t / kTmaStages;
      const int k0 = c0 + t * kTmaTileCells;
      const int k = k0 + (lane >> 2);
      const bool active = k < c1;
      int cells[NF + 1];
      int nblk = 0;
      int64_t off = 0;
      double xv[NF + 1][4];
      if (active) {
        nblk = sorted_blocks<NF>(m, k, cells);
        off = (__ldg(m.blk_start + k) - __ldg(m.blk_start + k0)) * (NL * NL) + int64_t(i) * nblk * NL;
#pragma unroll
        for (int s = 0; s < NF + 1; ++s)
          if (s < nblk) load_direction(p_cur, pv, par, beta, first, cells[s], xv[s]);
      }
      mbar_wait(full0 + 8 * stage, n & 1);
      double sum = 0.0;
      if (active) {
        const double* row = reinterpret_cast<const double*>(stage_base + stage * kTmaStageBytes) + off;
#pragma unroll
        for (int s = 0; s < NF + 1; ++s)
          if (s < nblk) {
            const double2 a = *reinterpret_cast<const double2*>(row + s * 4);
            const double2 b = *reinterpret_cast<const double2*>(row + s * 4 + 2);
            sum = fma(a.x, xv[s][0], sum); sum = fma(a.y, xv[s][1], sum);
            sum = fma(b.x, xv[s][2], sum); sum = fma(b.y, xv[s][3], sum);
          }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty0 + 8 * stage);
      if (active) {
        const int64_t r = int64_t(NL) * k + i;
        c.q[r] = sum;
        v[0] = fma(__ldg(p_cur + own_off + r), sum, v[0]);
      }
    }
  }
  grid_sum<1>(v, c.partial, &sc->ticket_a, [sc](const double(&w)[1]) { sc->red[0] = w[0]; });
}

// ---- TMA-staged SpMV, generic block size (P1 / P2 / Q2) ----------------------------------------------------------------
// Same pipeline as k_cg_spmv_tma with TC cells (TC * NL <= 32 rows) per warp tile.  Row blocks of NL = 3 and NL = 9 are
// only 8-byte aligned (72 / 648 bytes per block), so the producer copies from the enclosing 16-byte aligned range and the
// consumers skip the leading double.
template <int NF, int NL, int TC>
struct TmaCfg {
  static constexpr int kTileBytes = ((TC * (NF + 1) * NL * NL * 8 + 16 + 127) / 128) * 128;
  static constexpr int kStages = (200 * 1024 / kTileBytes) < 32 ? (200 * 1024 / kTileBytes) : 32;
  static constexpr int kConsumerWarps = NL >= 9 ? 12 : 16;
  static constexpr int kThreads = (kConsumerWarps + 1) * 32;
  static constexpr int kSmemBytes = kStages * kTileBytes + 2 * kStages * 8;
};

template <int NF, int NL, int TC>
__global__ void __launch_bounds__((TmaCfg<NF, NL, TC>::kThreads), 1)
    k_cg_spmv_tma_g(MeshView m, CgBuffers c, int par, int cells_per_cta) {
  using Cfg = TmaCfg<NF, NL, TC>;
  constexpr int S = Cfg::kStages;
  extern __shared__ __align__(128) unsigned char smem[];
  CgScalars* sc = c.sc;
  if (sc->done[par]) return;
  unsigned char* stage_base = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S * Cfg::kTileBytes);
  const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + S);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int c0 = blockIdx.x * cells_per_cta;
  const int c1 = min(c0 + cells_per_cta, m.n_own);
  const int n_tiles = c1 > c0 ? (c1 - c0 + TC - 1) / TC : 0;
  double v[1] = {0.0};
  if (warp == Cfg::kConsumerWarps) {
    // producer warp: in round n lane l (< S) feeds tile n * S + l into stage l.  All lanes walk the same rounds and meet
    // at the end of each one, so the warp reaches the final reduction converged.
    const int rounds = (n_tiles + S - 1) / S;
    for (int n = 0; n < rounds; ++n) {
      const int t = n * S + lane;
      if (lane < S && t < n_tiles) {
        if (n > 0) mbar_wait(empty0 + 8 * lane, (n - 1) & 1);
        const int k0 = c0 + t * TC, k1 = min(k0 + TC, c1);
        const int64_t e0 = __ldg(m.blk_start + k0) * (NL * NL), e1 = __ldg(m.blk_start + k1) * (NL * NL);
        const int64_t a0 = e0 & ~int64_t(1), a1 = (e1 + 1) & ~int64_t(1);  // 16-byte aligned element range
        const uint32_t bytes = uint32_t(a1 - a0) * 8;
        mbar_expect_tx(full0 + 8 * lane, bytes);
        bulk_g2s(smem_u32(stage_base + lane * Cfg::kTileBytes), c.values + a0, bytes, full0 + 8 * lane);
      }
      __syncwarp();
    }
  } else {
    const int64_t own_off = int64_t(m.own0) * NL;
    const int ci = lane / NL, i = lane - ci * NL;
    const double* p_cur = dir_in(c, par);
    for (int t = warp; t < n_tiles; t += Cfg::kConsumerWarps) {
      const int stage = t % S, n = t / S;
      const int k0 = c0 + t * TC;
      const int k = k0 + ci;
      const bool active = ci < TC && k < c1;
      int cells[NF + 1];
      int nblk = 0;
      int64_t off = 0;
      if (active) {
        nblk = sorted_blocks<NF>(m, k, cells);
        const int64_t e0 = __ldg(m.blk_start + k0) * (NL * NL);
        off = __ldg(m.blk_start + k) * (NL * NL) - (e0 & ~int64_t(1)) + int64_t(i) * nblk * NL;
        // touch the direction entries before waiting for the matrix tile: the gather then hits L1
#pragma unroll
        for (int s = 0; s < NF + 1; ++s)
          if (s < nblk) asm volatile("prefetch.global.L1 [%0];" ::"l"(p_cur + size_t(NL) * cells[s]));
      }
      mbar_wait(full0 + 8 * stage, n & 1);
      double sum = 0.0;
      if (active) {
        const double* row = reinterpret_cast<const double*>(stage_base + stage * Cfg::kTileBytes) + off;
#pragma unroll
        for (int s = 0; s < NF + 1; ++s)
          if (s < nblk) {
            const double* xs = p_cur + size_t(NL) * cells[s];
#pragma unroll
            for (int j = 0; j < NL; ++j) sum = fma(row[s * NL + j], __ldg(xs + j), sum);
          }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty0 + 8 * stage);
      if (active) {
        const int64_t r = int64_t(NL) * k + i;
        c.q[r] = sum;
        v[0] = fma(__ldg(p_cur + own_off + r), sum, v[0]);
      }
    }
  }
  grid_sum<1>(v, c.partial, &sc->ticket_a, [sc](const double(&w)[1]) { sc->red[0] = w[0]; });
}

template <int NF, int NL, int TC>
void launch_cg_spmv_tma_g(const MeshView& m, const CgBuffers& c, int parity, cudaStream_t s) {
  using Cfg = TmaCfg<NF, NL, TC>;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  static bool configured[64] = {};  // the opt-in to > 48 KB of dynamic shared memory is per device
  if (dev >= 0 && dev < 64 && !configured[dev]) {
    HDD_CUDA(cudaFuncSetAttribute(k_cg_spmv_tma_g<NF, NL, TC>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured[dev] = true;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (const char* e = std::getenv("HDD_SPMV_CTAS")) sms = std::max(1, std::atoi(e));  // tests: few CTAs => the ring wraps
  int cells_per_cta = (m.n_own + sms - 1) / sms;
  cells_per_cta = (cells_per_cta + TC - 1) / TC * TC;
  const int grid = (m.n_own + cells_per_cta - 1) / cells_per_cta;
  k_cg_spmv_tma_g<NF, NL, TC><<<grid, Cfg::kThreads, Cfg::kSmemBytes, s>>>(m, c, parity, cells_per_cta);
}

// ---- vector kernels ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kCgThreads) k_cg_init(int64_t rows, int64_t own_off, CgBuffers c) {
  double v[2] = {0.0, 0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < rows; t += stride) {
    const double b = c.b[t], z = c.dinv[t] * b;
    c.x[t] = 0.0;
    c.r[t] = b;
    c.p[own_off + t] = z;
    v[0] += b * z;
    v[1] += b * b;
  }
  CgScalars* sc = c.sc;
  grid_sum<2>(v, c.partial, &sc->ticket_a, [sc](const double(&w)[2]) {
    sc->red[1] = w[0];  // local r.z
    sc->red[2] = w[1];  // local b.b
  });
}

// block-Jacobi variant: one thread per cell, z = Dinv_T r_T with the inverted n_loc x n_loc diagonal block
template <int NL>
__global__ void __launch_bounds__(kCgThreads) k_cg_init_block(int64_t cells, int64_t own_off, CgBuffers c) {
  double v[2] = {0.0, 0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; k < cells; k += stride) {
    double b[NL], z[NL];
#pragma unroll
    for (int i = 0; i < NL; ++i) b[i] = c.b[NL * k + i];
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < NL; ++j) s = fma(__ldg(c.dinv_block + (NL * NL) * k + i * NL + j), b[j], s);
      z[i] = s;
    }
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      c.x[NL * k + i] = 0.0;
      c.r[NL * k + i] = b[i];
      c.z[NL * k + i] = z[i];
      c.p[own_off + NL * k + i] = z[i];
      v[0] = fma(b[i], z[i], v[0]);
      v[1] = fma(b[i], b[i], v[1]);
    }
  }
  CgScalars* sc = c.sc;
  grid_sum<2>(v, c.partial, &sc->ticket_a, [sc](const double(&w)[2]) {
    sc->red[1] = w[0];
    sc->red[2] = w[1];
  });
}

// after the (optional) all-reduce of red[1..2]
__global__ void k_cg_init_finish(CgScalars* sc) {
  sc->rz[0] = sc->red[1];
  sc->bb = sc->red[2];
  sc->rr = sc->red[2];
  sc->it[0] = 0;
  sc->done[0] = (sc->red[2] == 0.0 || sc->max_it <= 0) ? 1 : 0;
}

__global__ void __launch_bounds__(kCgThreads) k_cg_update(int64_t rows, int64_t own_off, CgBuffers c, int par) {
  CgScalars* sc = c.sc;
  if (sc->done[par]) return;
  const double alpha = sc->rz[par] / sc->red[0];
  double v[2] = {0.0, 0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  if ((rows & 3) == 0 && (own_off & 3) == 0) {
    // four rows per thread, 256-bit accesses
    const int64_t n4 = rows >> 2;
    for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < n4; t += stride) {
      double p[4], q[4], x[4], r[4], d[4];
      ld256_rw(dir_in(c, par) + own_off + 4 * t, p[0], p[1], p[2], p[3]);
      ld256_stream(c.q + 4 * t, q[0], q[1], q[2], q[3]);
      ld256_rw(c.x + 4 * t, x[0], x[1], x[2], x[3]);
      ld256_rw(c.r + 4 * t, r[0], r[1], r[2], r[3]);
      ld256_stream(c.dinv + 4 * t, d[0], d[1], d[2], d[3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        x[j] = fma(alpha, p[j], x[j]);
        r[j] = fma(-alpha, q[j], r[j]);
        const double z = d[j] * r[j];
        v[0] = fma(r[j], z, v[0]);
        v[1] = fma(r[j], r[j], v[1]);
      }
      st256(c.x + 4 * t, x[0], x[1], x[2], x[3]);
      st256(c.r + 4 * t, r[0], r[1], r[2], r[3]);
    }
  } else {
    for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < rows; t += stride) {
      c.x[t] = fma(alpha, dir_in(c, par)[own_off + t], c.x[t]);
      const double r = fma(-alpha, c.q[t], c.r[t]);
      c.r[t] = r;
      const double z = c.dinv[t] * r;
      v[0] = fma(r, z, v[0]);
      v[1] = fma(r, r, v[1]);
    }
  }
  grid_sum<2>(v, c.partial, &sc->ticket_b, [sc](const double(&w)[2]) {
    sc->red[1] = w[0];
    sc->red[2] = w[1];
  });
}

template <int NL>
__global__ void __launch_bounds__(kCgThreads) k_cg_update_block(int64_t cells, int64_t own_off, CgBuffers c, int par) {
  CgScalars* sc = c.sc;
  if (sc->done[par]) return;
  const double alpha = sc->rz[par] / sc->red[0];
  double v[2] = {0.0, 0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; k < cells; k += stride) {
    double p[NL], q[NL], x[NL], r[NL], z[NL], D[NL * NL];
    if constexpr (NL == 4) {
      ld256_rw(dir_in(c, par) + own_off + 4 * k, p[0], p[1], p[2], p[3]);
      ld256_stream(c.q + 4 * k, q[0], q[1], q[2], q[3]);
      ld256_rw(c.x + 4 * k, x[0], x[1], x[2], x[3]);
      ld256_rw(c.r + 4 * k, r[0], r[1], r[2], r[3]);
#pragma unroll
      for (int i = 0; i < 4; ++i) ld256_stream(c.dinv_block + 16 * k + 4 * i, D[4 * i], D[4 * i + 1], D[4 * i + 2], D[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < NL; ++i) {
        p[i] = dir_in(c, par)[own_off + NL * k + i]; q[i] = c.q[NL * k + i]; x[i] = c.x[NL * k + i]; r[i] = c.r[NL * k + i];
      }
#pragma unroll
      for (int i = 0; i < NL * NL; ++i) D[i] = __ldg(c.dinv_block + (NL * NL) * k + i);
    }
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      x[i] = fma(alpha, p[i], x[i]);
      r[i] = fma(-alpha, q[i], r[i]);
    }
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < NL; ++j) s = fma(D[i * NL + j], r[j], s);
      z[i] = s;
      v[0] = fma(r[i], s, v[0]);
      v[1] = fma(r[i], r[i], v[1]);
    }
    if constexpr (NL == 4) {
      st256(c.x + 4 * k, x[0], x[1], x[2], x[3]);
      st256(c.r + 4 * k, r[0], r[1], r[2], r[3]);
      st256(c.z + 4 * k, z[0], z[1], z[2], z[3]);
    } else {
#pragma unroll
      for (int i = 0; i < NL; ++i) { c.x[NL * k + i] = x[i]; c.r[NL * k + i] = r[i]; c.z[NL * k + i] = z[i]; }
    }
  }
  grid_sum<2>(v, c.partial, &sc->ticket_b, [sc](const double(&w)[2]) {
    sc->red[1] = w[0];
    sc->red[2] = w[1];
  });
}

// p = z + beta p with z = dinv r (diagonal / identity) or the stored z (block Jacobi); also advances the CG state
__global__ void __launch_bounds__(kCgThreads) k_cg_direction(int64_t rows, int64_t own_off, CgBuffers c, int par) {
  CgScalars* sc = c.sc;
  const int done = sc->done[par];
  if (!done) {
    const double beta = sc->red[1] / sc->rz[par];
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    const bool stored_z = c.z != nullptr;
    const double* pin = dir_in(c, par);
    double* pout = dir_out(c, par);
    if ((rows & 3) == 0 && (own_off & 3) == 0) {
      const int64_t n4 = rows >> 2;
      for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < n4; t += stride) {
        double p[4], z[4];
        ld256_rw(pin + own_off + 4 * t, p[0], p[1], p[2], p[3]);
        if (stored_z) {
          ld256_rw(c.z + 4 * t, z[0], z[1], z[2], z[3]);
        } else {
          double r[4];
          ld256_rw(c.r + 4 * t, r[0], r[1], r[2], r[3]);
          ld256_stream(c.dinv + 4 * t, z[0], z[1], z[2], z[3]);
#pragma unroll
          for (int j = 0; j < 4; ++j) z[j] *= r[j];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) p[j] = fma(beta, p[j], z[j]);
        st256(pout + own_off + 4 * t, p[0], p[1], p[2], p[3]);
      }
    } else {
      for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < rows; t += stride) {
        const double z = stored_z ? c.z[t] : c.dinv[t] * c.r[t];
        pout[own_off + t] = fma(beta, pin[own_off + t], z);
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (done) {
      sc->rz[par ^ 1] = sc->rz[par];
      sc->it[par ^ 1] = sc->it[par];
      sc->done[par ^ 1] = 1;
    } else {
      const int it = sc->it[par] + 1;
      sc->rz[par ^ 1] = sc->red[1];
      sc->rr = sc->red[2];
      sc->it[par ^ 1] = it;
      sc->done[par ^ 1] = (sc->red[2] <= sc->tol2 * sc->bb || it >= sc->max_it) ? 1 : 0;
    }
  }
}

// inverse of the n_loc x n_loc diagonal block of every owned cell (Gauss-Jordan, the blocks are s.p.d.)
template <int NF, int NL>
__global__ void k_invert_diag_blocks(MeshView m, const double* __restrict__ values, double* __restrict__ dinv_block) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m.n_own) return;
  int nb[NF];
  load_neigh<NF>(m.neigh, k, nb);
  const int self = m.own0 + k;
  const int nblk = block_count<NF>(nb);
  const int slot = block_slot<NF>(self, nb, self);
  const double* row0 = values + m.blk_start[k] * (NL * NL);
  double A[NL][NL], I[NL][NL];
#pragma unroll
  for (int i = 0; i < NL; ++i)
#pragma unroll
    for (int j = 0; j < NL; ++j) {
      A[i][j] = row0[size_t(i) * nblk * NL + slot * NL + j];
      I[i][j] = i == j ? 1.0 : 0.0;
    }
#pragma unroll
  for (int c = 0; c < NL; ++c) {
    const double ip = 1.0 / A[c][c];
#pragma unroll
    for (int j = 0; j < NL; ++j) { A[c][j] *= ip; I[c][j] *= ip; }
#pragma unroll
    for (int i = 0; i < NL; ++i)
      if (i != c) {
        const double f = A[i][c];
#pragma unroll
        for (int j = 0; j < NL; ++j) { A[i][j] = fma(-f, A[c][j], A[i][j]); I[i][j] = fma(-f, I[c][j], I[i][j]); }
      }
  }
#pragma unroll
  for (int i = 0; i < NL; ++i)
#pragma unroll
    for (int j = 0; j < NL; ++j) dinv_block[size_t(NL * NL) * k + i * NL + j] = 0.5 * (I[i][j] + I[j][i]);
}

// a15: pure-Neumann fix of ContainerBasedDefault::uncached_solve (discretizations/base.hh:337-345): unit_row(0) and
// rhs[0] = 0.  Done symmetrically (row and column 0) so that CG stays applicable; with rhs[0] = 0 both give x_0 = 0
// and the same remaining system.  One warp, cell 0 and its neighbours only.
template <int NF, int NL>
__global__ void k_unit_row_col0(MeshView m, double* __restrict__ vals, double* __restrict__ b) {
  if (threadIdx.x != 0 || blockIdx.x != 0 || m.n_own == 0 || m.own0 != 0) return;
  int nb[NF];
  load_neigh<NF>(m.neigh, 0, nb);
  const int nblk = block_count<NF>(nb);
  double* row0 = vals + m.blk_start[0] * (NL * NL);
  const int self_slot = block_slot<NF>(0, nb, 0);
  for (int t = 0; t < nblk * NL; ++t) row0[t] = 0.0;                                  // row 0
  for (int i = 0; i < NL; ++i) row0[size_t(i) * nblk * NL + self_slot * NL + 0] = 0.0;  // column 0 inside cell 0
  row0[self_slot * NL] = 1.0;
  for (int f = 0; f < NF; ++f) {
    const int n = nb[f];
    if (n < 0 || n >= m.n_own) continue;
    int nn[NF];
    load_neigh<NF>(m.neigh, n, nn);
    const int cnt = block_count<NF>(nn);
    const int slot = block_slot<NF>(n, nn, 0);
    double* r = vals + m.blk_start[n] * (NL * NL);
    for (int i = 0; i < NL; ++i) r[size_t(i) * cnt * NL + slot * NL + 0] = 0.0;        // column 0 in the neighbour's rows
  }
  b[0] = 0.0;
}

__global__ void __launch_bounds__(kCgThreads) k_sum(const double* __restrict__ x, int64_t n, double* partial,
                                                    unsigned int* ticket, double* out) {
  double v[1] = {0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < n; t += stride) v[0] += x[t];
  grid_sum<1>(v, partial, ticket, [out](const double(&w)[1]) { *out = w[0]; });
}

__global__ void __launch_bounds__(kCgThreads) k_residual_norms(const double* __restrict__ b, const double* __restrict__ q,
                                                              const double* __restrict__ x, int64_t n, double* partial,
                                                              CgScalars* sc) {
  double v[3] = {0.0, 0.0, 0.0};
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const double bi = b[i], d = bi - q[i], xi = x[i];
    v[0] = fma(d, d, v[0]);
    v[1] = fma(bi, bi, v[1]);
    v[2] = fma(xi, xi, v[2]);
  }
  grid_sum<3>(v, partial, &sc->ticket_a, [sc](const double(&w)[3]) { sc->red[0] = w[0]; sc->red[1] = w[1]; sc->red[2] = w[2]; });
}

// *out = max |v[i]| (out must hold 0 on entry; non-negative doubles order like their bit patterns)
__global__ void __launch_bounds__(kCgThreads) k_abs_max(const double* __restrict__ v, int64_t n, double* out) {
  double m = 0.0;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) m = fmax(m, fabs(v[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned long long*>(out), (unsigned long long)__double_as_longlong(m));
}

__global__ void k_shift(double* __restrict__ x, int64_t n, const double* __restrict__ sum, double inv_count) {
  const double mean = *sum * inv_count;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < n; t += stride) x[t] -= mean;
}

__global__ void k_pack(const double* __restrict__ v, const int32_t* __restrict__ cells, int64_t n, int nd,
                       double* __restrict__ out) {
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < n; t += stride) {
    const int64_t k = t / nd;
    out[t] = v[int64_t(cells[k]) * nd + (t - k * nd)];
  }
}

inline int cg_grid(int64_t items) {
  const int64_t need = (items + kCgThreads - 1) / kCgThreads;
  return int(std::max<int64_t>(1, std::min<int64_t>(need, kMaxBlocks)));
}

}  // namespace

bool cg_spmv_uses_tma(const MeshView& m) {
  return m.kind == HDD_CUBE2D && m.nl == 4 && m.n_own >= 148 * kTmaTileCells;
}

int cg_partial_capacity() { return 3 * kMaxBlocks; }

void launch_spmv(const MeshView& m, const double* values, const double* x_local, double* y, cudaStream_t s) {
  const int64_t rows = int64_t(m.n_own) * m.nl;
  if (rows == 0) return;
  dispatch_block(m, [&](auto nf, auto nl) {
    k_spmv<decltype(nf)::value, decltype(nl)::value><<<cg_grid(rows), kCgThreads, 0, s>>>(m, values, x_local, y);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_invert_diag_blocks(const MeshView& m, const double* values, double* dinv_block, cudaStream_t s) {
  if (m.n_own == 0) return;
  dispatch_block(m, [&](auto nf, auto nl) {
    k_invert_diag_blocks<decltype(nf)::value, decltype(nl)::value><<<(m.n_own + 127) / 128, 128, 0, s>>>(m, values, dinv_block);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_cg_init(const MeshView& m, const CgBuffers& c, double precision, int max_it, cudaStream_t s) {
  const int64_t rows = int64_t(m.n_own) * m.nl;
  CgScalars h{};
  h.tol2 = precision * precision;
  h.max_it = max_it;
  HDD_CUDA(cudaMemcpyAsync(c.sc, &h, sizeof(h), cudaMemcpyHostToDevice, s));
  if (c.dinv_block) {
    dispatch_nl(m.nl, [&](auto nl) {
      k_cg_init_block<decltype(nl)::value><<<cg_grid(m.n_own), kCgThreads, 0, s>>>(m.n_own, int64_t(m.own0) * m.nl, c);
    });
  } else {
    k_cg_init<<<cg_grid(rows), kCgThreads, 0, s>>>(rows, int64_t(m.own0) * m.nl, c);
  }
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_cg_init_finish(const MeshView&, const CgBuffers& c, cudaStream_t s) {
  k_cg_init_finish<<<1, 1, 0, s>>>(c.sc);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_cg_spmv(const MeshView& m, const CgBuffers& c, int parity, cudaStream_t s, const PeerView* peer) {
  const int64_t rows = int64_t(m.n_own) * m.nl;
  if (cg_spmv_uses_tma(m)) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    static bool configured[64] = {};  // the opt-in to > 48 KB of dynamic shared memory is per device
    if (dev >= 0 && dev < 64 && !configured[dev]) {
      HDD_CUDA(cudaFuncSetAttribute(k_cg_spmv_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, kTmaSmemBytes));
      configured[dev] = true;
    }
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (const char* e = std::getenv("HDD_SPMV_CTAS")) sms = std::max(1, std::atoi(e));  // tests: few CTAs => the ring wraps
    int cells_per_cta = (m.n_own + sms - 1) / sms;
    cells_per_cta = (cells_per_cta + kTmaTileCells - 1) / kTmaTileCells * kTmaTileCells;
    const int grid = (m.n_own + cells_per_cta - 1) / cells_per_cta;
    PeerView pv{};
    if (peer) pv = *peer;
    k_cg_spmv_tma<<<grid, kTmaThreads, kTmaSmemBytes, s>>>(m, c, parity, cells_per_cta, pv);
  } else if (!peer && m.n_own >= 1024 && !(m.nf == 4 && m.nl == 4)) {
    if (m.nf == 3 && m.nl == 3) launch_cg_spmv_tma_g<3, 3, 10>(m, c, parity, s);
    else if (m.nf == 3 && m.nl == 6) launch_cg_spmv_tma_g<3, 6, 5>(m, c, parity, s);
    else if (m.nf == 4 && m.nl == 9) launch_cg_spmv_tma_g<4, 9, 3>(m, c, parity, s);
    else HDD_THROW(HDD_ERR_INTERNAL, "unsupported block shape nf = " << m.nf << ", nl = " << m.nl);
  } else {
    dispatch_block(m, [&](auto nf, auto nl) {
      k_cg_spmv<decltype(nf)::value, decltype(nl)::value><<<cg_grid(rows), kCgThreads, 0, s>>>(m, c, parity);
    });
  }
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_cg_update(const MeshView& m, const CgBuffers& c, int parity, cudaStream_t s) {
  const int64_t rows = int64_t(m.n_own) * m.nl;
  if (c.dinv_block) {
    dispatch_nl(m.nl, [&](auto nl) {
      k_cg_update_block<decltype(nl)::value><<<cg_grid(m.n_own), kCgThreads, 0, s>>>(m.n_own, int64_t(m.own0) * m.nl, c, parity);
    });
  } else {
    k_cg_update<<<cg_grid((rows + 3) / 4), kCgThreads, 0, s>>>(rows, int64_t(m.own0) * m.nl, c, parity);
  }
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_cg_direction(const MeshView& m, const CgBuffers& c, int parity, cudaStream_t s) {
  const int64_t rows = int64_t(m.n_own) * m.nl;
  k_cg_direction<<<cg_grid((rows + 3) / 4), kCgThreads, 0, s>>>(rows, int64_t(m.own0) * m.nl, c, parity);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_unit_row_col0(const MeshView& m, double* values, double* b, cudaStream_t s) {
  dispatch_block(m, [&](auto nf, auto nl) {
    k_unit_row_col0<decltype(nf)::value, decltype(nl)::value><<<1, 32, 0, s>>>(m, values, b);
  });
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

void launch_subtract_mean(double* x, int64_t n, double* partial, CgScalars* sc, cudaStream_t s) {
  if (n == 0) return;
  k_sum<<<cg_grid(n), kCgThreads, 0, s>>>(x, n, partial, &sc->ticket_a, &sc->red[3]);
  k_shift<<<cg_grid(n), kCgThreads, 0, s>>>(x, n, &sc->red[3], 1.0 / double(n));
  count_launch(2);
  HDD_CUDA(cudaGetLastError());
}

void launch_residual_norms(const double* b, const double* q, const double* x, int64_t n, const double* values, int64_t nnz,
                           double* partial, CgScalars* sc, cudaStream_t s) {
  k_residual_norms<<<cg_grid(n), kCgThreads, 0, s>>>(b, q, x, n, partial, sc);
  HDD_CUDA(cudaMemsetAsync(&sc->red[3], 0, sizeof(double), s));
  k_abs_max<<<cg_grid(nnz), kCgThreads, 0, s>>>(values, nnz, &sc->red[3]);
  count_launch(2);
}

void launch_pack(const double* v_local, const int32_t* cells, int64_t n_cells, int nd, double* out, cudaStream_t s) {
  const int64_t n = n_cells * nd;
  if (n == 0) return;
  k_pack<<<int(std::min<int64_t>((n + 255) / 256, 1024)), 256, 0, s>>>(v_local, cells, n, nd, out);
  count_launch();
  HDD_CUDA(cudaGetLastError());
}

}  // namespace hdd
