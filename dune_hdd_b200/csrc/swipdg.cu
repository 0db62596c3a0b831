// hdd_swipdg: the discretization handle - problem localisation, init() (pattern + assembly of all affine parts),
// freeze + CG solve, operator parts / BlockSWIPDG views, estimator dispatch.
// Mirrors dune/hdd/linearelliptic/discretizations/{swipdg,block-swipdg,base}.hh and estimators/{swipdg,block-swipdg}.hh.
#include <algorithm>
#include <cmath>
#include <cstring>

#include <dlfcn.h>

#include "handles.hpp"

using namespace hdd;

hdd_swipdg::~hdd_swipdg() {
  if (p2p_ready && mesh) {
    // The neighbours read r / p / p_alt of this rank through their own IPC mappings.  Nobody frees an exported buffer
    // before every rank has finished its kernels and closed its mappings: drain the stream, close, then meet the other
    // ranks in one all-reduce (destruction of a distributed discretization is collective, like its construction).
    cudaStreamSynchronize(mesh->stream);
    for (void* p : ipc_opened) cudaIpcCloseMemHandle(p);
    ipc_opened.clear();
    if (mesh->world > 1 && mesh->comm && sc.p) {
      try {
        hdd::Nccl::get().all_reduce_sum(&sc.p->red[0], 1, mesh->comm, mesh->stream);
        cudaStreamSynchronize(mesh->stream);
      } catch (...) {
      }
    }
  }
  for (void* p : ipc_opened) cudaIpcCloseMemHandle(p);
  if (sc_host) cudaFreeHost(sc_host);
  if (mg) hdd::mg_release(mg);
  for (auto& g : cg_graph)
    if (g.exec) cudaGraphExecDestroy(g.exec);
}

namespace hdd {

void require_init(const hdd_swipdg* h) {
  if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
  if (!h->initialized)
    HDD_THROW(HDD_ERR_USING_THIS_WRONG, "The user has to call init() before calling any other method!");
}

// map_parameter + type check of uncached_solve (discretizations/base.hh:333-334)
void check_mu(const hdd_swipdg* h, const double* mu, int mu_size, const char* name) {
  const bool parametric = h->factor.parametric() || h->force.parametric() || h->dirichlet.parametric() || h->neumann.parametric();
  if (parametric) {
    if (!mu || mu_size != h->parameter_size)
      HDD_THROW(HDD_ERR_WRONG_PARAMETER_TYPE, name << " has size " << (mu ? mu_size : 0) << " vs. parameter type {"
                                                   << h->parameter_name << ": " << h->parameter_size << "}");
  } else if (mu && mu_size != 0) {
    HDD_THROW(HDD_ERR_WRONG_PARAMETER_TYPE, name << " has size " << mu_size << " vs. empty parameter type");
  }
}

double eval_coef(const Program& p, const double* mu, int mu_size) {
  double v[4] = {0, 0, 0, 0};
  for (int k = 0; k < mu_size && k < 4; ++k) v[k] = mu[k];
  return eval_program(p, v);
}

DevCombo make_combo(const hdd_swipdg* h, const AffineFn& f, const double* mu, int mu_size) {
  DevCombo c{};
  int order = 0;
  for (size_t q = 0; q < f.comps.size(); ++q) {
    c.theta[c.n] = eval_coef(f.coef_prog[q], mu, mu_size);
    c.idx[c.n++] = f.comps[q].idx;
    order = std::max(order, f.comps[q].order);
  }
  if (f.has_affine()) {
    c.theta[c.n] = 1.0;
    c.idx[c.n++] = f.affine.idx;
    order = std::max(order, f.affine.order);
  }
  c.order = order;
  return c;
}

}  // namespace hdd

namespace {

constexpr double kPi = 3.14159265358979323846264338327950288;

FnRef add_function(hdd_swipdg* h, const hdd_function& f, const char* what) {
  hdd_mesh* m = h->mesh;
  DevFn d{};
  d.kind = f.kind;
  d.order = f.order;
  d.value = f.value;
  d.cell = nullptr;
  d.prog.n_ops = 0;
  d.separable = 0;
  d.px.n_ops = 0;
  d.py.n_ops = 0;
  FnRef r;
  r.order = f.order;
  r.kind = f.kind;
  if (f.order < 0 || f.order > 12) HDD_THROW(HDD_ERR_WRONG_INPUT, what << ": unsupported order " << f.order);
  switch (f.kind) {
    case HDD_FN_CONSTANT:
      r.zero = (f.value == 0.0);
      break;
    case HDD_FN_CELLWISE: {
      if (!f.cell_values) HDD_THROW(HDD_ERR_WRONG_INPUT, what << ": cell_values is NULL");
      h->fn_cell_storage.emplace_back(new DevBuf<double>);
      if (m->whole) {  // local numbering = global numbering: upload the caller's array as it is
        h->fn_cell_storage.back()->upload(f.cell_values, size_t(m->n_loc), m->stream);
      } else {
        std::vector<double> loc(size_t(m->n_loc));
        for (int32_t lc = 0; lc < m->n_loc; ++lc) loc[size_t(lc)] = f.cell_values[m->gid(lc)];
        h->fn_cell_storage.back()->upload(loc.data(), loc.size(), m->stream);
      }
      HDD_CUDA(cudaStreamSynchronize(m->stream));
      d.cell = h->fn_cell_storage.back()->p;
      break;
    }
    case HDD_FN_EXPRESSION:
      if (!f.expression) HDD_THROW(HDD_ERR_WRONG_INPUT, what << ": expression is NULL");
      d.prog = compile_expression(f.expression, "x");
      d.separable = compile_separable(f.expression, "x", d.px, d.py) ? 1 : 0;
      {
        static const bool fast_on = [] { const char* e = std::getenv("HDD_EXPR_FAST"); return !(e && e[0] == '0'); }();
        if (fast_on) compile_fast(f.expression, "x", d.fast);
      }
      break;
    default:
      HDD_THROW(HDD_ERR_WRONG_INPUT, what << ": unknown function kind " << f.kind);
  }
  r.idx = int(h->fn_host.size());
  r.separable = d.separable != 0;
  h->fn_host.push_back(d);
  return r;
}

AffineFn add_affine(hdd_swipdg* h, const hdd_affine_function& a, const char* what) {
  AffineFn out;
  if (a.n_components < 0 || a.n_components > kMaxParts - 1)
    HDD_THROW(HDD_ERR_WRONG_INPUT, what << ": unsupported number of components " << a.n_components);
  for (int q = 0; q < a.n_components; ++q) {
    if (!a.components || !a.coefficients || !a.coefficients[q])
      HDD_THROW(HDD_ERR_WRONG_INPUT, what << ": component arrays are NULL");
    out.comps.push_back(add_function(h, a.components[q], what));
    out.coef_expr.emplace_back(a.coefficients[q]);
    out.coef_prog.push_back(compile_expression(a.coefficients[q], h->parameter_name.empty() ? "mu" : h->parameter_name));
  }
  if (a.affine_part) out.affine = add_function(h, *a.affine_part, what);
  return out;
}

void assemble_all(hdd_swipdg* h) {
  hdd_mesh* m = h->mesh;
  const MeshView v = h->view();
  cudaStream_t s = m->stream;
  for (auto& part : h->lhs_comps) launch_assemble_lhs(v, h->fn_h(part.factor), part.factor.kind, part.factor.order, h->polorder, part.values.p, s);
  if (h->lhs_affine)
    launch_assemble_lhs(v, h->fn_h(h->lhs_affine->factor), h->lhs_affine->factor.kind, h->lhs_affine->factor.order, h->polorder,
                        h->lhs_affine->values.p, s);
  TensorGridView tg;
  if (m->sx > 0) {
    tg.nx = m->sx;
    tg.ny = m->sy;
    tg.cell_v0 = m->cell_v0.p;
    const size_t need = size_t(m->sx + m->sy) * (2 + h->polorder + 1);
    if (h->rhs_scratch.n < need) h->rhs_scratch.alloc(need);
    tg.scratch = h->rhs_scratch.p;
  }
  auto do_vec = [&](VectorPart& part) {
    // the first volume term overwrites the vector; only parts without one need the memset
    bool written = false;
    for (const RhsTerm& t : part.terms) written |= (t.kind == 0 && !t.f.zero);
    if (!written) part.values.zero(s);
    bool first = true;
    for (const RhsTerm& t : part.terms)
      if (t.kind == 0 && !t.f.zero) {
        launch_rhs_volume(v, h->fn_h(t.f), t.f.order, t.f.separable, h->polorder, !first, &tg, part.values.p, s);
        first = false;
      }
    for (const RhsTerm& t : part.terms) {
      if (t.kind == 0) {
        continue;
      } else if (t.kind == 2) {
        if (!t.f.zero) launch_rhs_neumann(v, h->fn_h(t.f), t.f.order, h->polorder, part.values.p, s);
      } else {
        if (!t.f.zero && !t.g.zero)
          launch_rhs_dirichlet(v, h->fn_h(t.f), t.f.order, h->fn_h(t.g), t.g.order, h->polorder, part.values.p, s);
      }
    }
  };
  for (auto& part : h->rhs_comps) do_vec(part);
  if (h->rhs_affine) do_vec(*h->rhs_affine);
}

// A(mu) = A_aff + sum theta_q A_q; returns the value array the solver should read
const double* freeze_lhs(hdd_swipdg* h, const double* mu, int mu_size) {
  if (h->lhs_comps.empty()) {
    if (!h->lhs_affine) HDD_THROW(HDD_ERR_WRONG_INPUT, "the diffusion factor is empty");
    return h->lhs_affine->values.p;
  }
  FreezeArgs a{};
  for (auto& part : h->lhs_comps) {
    a.theta[a.n] = eval_coef(part.coef_prog, mu, mu_size);
    a.part[a.n++] = part.values.p;
  }
  if (h->lhs_affine) {
    a.theta[a.n] = 1.0;
    a.part[a.n++] = h->lhs_affine->values.p;
  }
  if (!h->frozen.p) h->frozen.alloc(size_t(h->nnz));
  launch_freeze(a, h->frozen.p, h->nnz, h->mesh->stream);
  return h->frozen.p;
}

void freeze_rhs(hdd_swipdg* h, const double* mu, int mu_size) {
  FreezeArgs a{};
  for (auto& part : h->rhs_comps) {
    a.theta[a.n] = eval_coef(part.coef_prog, mu, mu_size);
    a.part[a.n++] = part.values.p;
  }
  if (h->rhs_affine) {
    a.theta[a.n] = 1.0;
    a.part[a.n++] = h->rhs_affine->values.p;
  }
  if (!h->b.p) h->b.alloc(size_t(h->n_rows));
  if (a.n == 0) { h->b.zero(h->mesh->stream); return; }
  launch_freeze(a, h->b.p, h->n_rows, h->mesh->stream);
}

void ensure_solve_workspace(hdd_swipdg* h) {
  hdd_mesh* m = h->mesh;
  const size_t rows = size_t(h->n_rows), loc = size_t(m->n_loc) * h->nl;
  if (!h->x.p) {
    h->dinv.alloc(rows);
    h->x.alloc(rows);
    h->r.alloc(rows);
    h->q.alloc(rows);
    h->p.alloc(loc);
    h->p.zero(m->stream);
    h->partial.alloc(size_t(cg_partial_capacity()));
    h->sc.alloc(1);
    HDD_CUDA(cudaMallocHost(reinterpret_cast<void**>(&h->sc_host), sizeof(CgScalars)));
  }
}

// ---- peer-memory SpMV set-up ------------------------------------------------------------------------------------
// Each rank publishes its residual and its two direction buffers through CUDA IPC; neighbours map them and the SpMV
// kernel reads halo entries straight from the owner's HBM over NVLink.  Collective: every rank must call it, and the
// outcome (all ranks succeeded?) is agreed on with an all-reduce so that nobody falls back alone.
struct IpcRecord {
  cudaIpcMemHandle_t handle[3];
  uint64_t offset[3];  // pointer - allocation base (cudaMalloc may sub-allocate)
};

uint64_t allocation_offset(const void* ptr) {
  typedef int (*get_range_t)(unsigned long long*, size_t*, unsigned long long);
  static get_range_t fn = [] {
    void* lib = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    return lib ? reinterpret_cast<get_range_t>(dlsym(lib, "cuMemGetAddressRange_v2")) : nullptr;
  }();
  if (!fn) HDD_THROW(HDD_ERR_DEVICE, "libcuda.so.1 / cuMemGetAddressRange_v2 not available");
  unsigned long long base = 0;
  size_t size = 0;
  if (fn(&base, &size, reinterpret_cast<unsigned long long>(ptr)) != 0) HDD_THROW(HDD_ERR_DEVICE, "cuMemGetAddressRange failed");
  return uint64_t(reinterpret_cast<unsigned long long>(ptr) - base);
}

bool p2p_wanted() {
  static const bool on = [] { const char* e = std::getenv("HDD_P2P"); return !(e && e[0] == '0'); }();
  return on;
}

// collective yes / no: true iff every rank passes ok = true (one all-reduce, one host synchronisation)
static bool all_ranks_ok(hdd_mesh* m, bool ok) {
  cudaStream_t s = m->stream;
  DevBuf<double> flag;
  double f = ok ? 0.0 : 1.0;
  flag.upload(&f, 1, s);
  Nccl::get().all_reduce_sum(flag.p, 1, m->comm, s);
  HDD_CUDA(cudaMemcpyAsync(&f, flag.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  HDD_CUDA(cudaStreamSynchronize(s));
  return f == 0.0;
}

// Every step that can fail on one rank alone is followed by a collective agreement before the next collective, so the
// ranks always issue the same sequence of NCCL calls: (1) local allocations and IPC export, agree; (2) all-gather of the
// handles, open the neighbours' handles, agree.  A failure anywhere makes every rank fall back to the NCCL halo exchange.
bool setup_p2p(hdd_swipdg* h) {
  hdd_mesh* m = h->mesh;
  if (h->p2p_ready) return true;
  if (h->p2p_failed) return false;
  cudaStream_t s = m->stream;
  Nccl& nc = Nccl::get();
  const size_t loc = size_t(m->n_loc) * h->nl;
  // (1) local work only
  bool ok = true;
  IpcRecord mine{};
  try {
    if (m->world > kMaxPeers) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "peer-memory SpMV supports at most " << kMaxPeers << " ranks");
    h->p_alt.alloc(loc);
    h->p_alt.zero(s);
    h->dinv_local.alloc(loc);
    h->dinv_local.zero(s);
    const void* ptrs[3] = {h->r.p, h->p.p, h->p_alt.p};
    for (int k = 0; k < 3; ++k) {
      HDD_CUDA(cudaIpcGetMemHandle(&mine.handle[k], const_cast<void*>(ptrs[k])));
      mine.offset[k] = allocation_offset(ptrs[k]);
    }
  } catch (const Error& e) {
    set_last_error(e.what());
    cudaGetLastError();
    ok = false;
  }
  if (!all_ranks_ok(m, ok)) {
    h->p2p_failed = true;
    h->p_alt.release();
    return false;
  }
  // (2) every rank takes part in the all-gather; opening a handle can fail locally again
  std::vector<IpcRecord> all(size_t(m->world));
  {
    DevBuf<unsigned char> send, recv;
    send.upload(reinterpret_cast<const unsigned char*>(&mine), sizeof(mine), s);
    recv.alloc(sizeof(IpcRecord) * size_t(m->world));
    nc.all_gather_bytes(send.p, recv.p, sizeof(IpcRecord), m->comm, s);
    HDD_CUDA(cudaMemcpyAsync(all.data(), recv.p, sizeof(IpcRecord) * size_t(m->world), cudaMemcpyDeviceToHost, s));
    HDD_CUDA(cudaStreamSynchronize(s));
  }
  PeerView pv{};
  pv.own0 = m->own0;
  pv.n_own = m->n_own;
  pv.halo_peer = m->halo_peer.p;
  pv.halo_rcell = m->halo_rcell.p;
  pv.dinv_local = h->dinv_local.p;
  for (const HaloPeer& peer : m->peers) {
    void* opened[3] = {nullptr, nullptr, nullptr};
    for (int k = 0; k < 3 && ok; ++k) {
      if (cudaIpcOpenMemHandle(&opened[k], all[size_t(peer.rank)].handle[k], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        ok = false;
        break;
      }
      h->ipc_opened.push_back(opened[k]);
    }
    if (!ok) break;
    pv.r[peer.rank] = reinterpret_cast<const double*>(static_cast<char*>(opened[0]) + all[size_t(peer.rank)].offset[0]);
    pv.p[0][peer.rank] = reinterpret_cast<const double*>(static_cast<char*>(opened[1]) + all[size_t(peer.rank)].offset[1]);
    pv.p[1][peer.rank] = reinterpret_cast<const double*>(static_cast<char*>(opened[2]) + all[size_t(peer.rank)].offset[2]);
    pv.own0_of[peer.rank] = m->rank_own0[size_t(peer.rank)];
  }
  if (!all_ranks_ok(m, ok)) {
    // nobody uses the mappings: close what was opened; the exported buffers stay allocated until every rank has passed
    // the agreement above, which it has
    for (void* p : h->ipc_opened) cudaIpcCloseMemHandle(p);
    h->ipc_opened.clear();
    h->p2p_failed = true;
    h->p_alt.release();
    return false;
  }
  pv.enabled = 1;
  h->peer_view = pv;
  h->p2p_ready = true;
  return true;
}

// the solver types in the order hdd_solver_types lists their canonical names, with the other spellings hdd_solve accepts
struct SolverTypeName {
  SolverType type;
  const char* name;
  const char* aliases[5];  // unused entries nullptr
};
const SolverTypeName kSolverTypes[] = {
    {SolverType::diagonal, "cg.diagonal", {"", "cg", "cg.jacobi", "cg.diagonal.lower", "cg.diagonal.upper"}},
    {SolverType::blockdiagonal, "cg.blockdiagonal", {"cg.blockjacobi"}},
    {SolverType::identity, "cg.identity", {"cg.identity.lower", "cg.identity.upper"}},
    {SolverType::mg, "cg.mg", {"cg.multigrid"}},
    {SolverType::mg2, "cg.mg2", {"cg.multigrid2"}},
    {SolverType::mg2_simplex, "cg.mg2.simplex", {"cg.multigrid2.simplex"}},
};

SolverType parse_solver_type(const char* type) {
  const std::string t = type ? type : "";
  for (const SolverTypeName& e : kSolverTypes) {
    if (t == e.name) return e.type;
    for (const char* a : e.aliases)
      if (a && t == a) return e.type;
  }
  HDD_THROW(HDD_ERR_WRONG_INPUT, "solver type '" << t << "' is not one of solver_types()");
}

// Pymor::AffinelyDecomposableFunctionInterface::alpha / gamma (call sites estimators/block-swipdg.hh:778-781):
// min / max over the components of theta_q(mu1) / theta_q(mu2); 1 for non-parametric functions.
void alpha_gamma(const hdd_swipdg* h, const double* mu1, const double* mu2, int mu_size, double& alpha, double& gamma) {
  alpha = 1.0;
  gamma = 1.0;
  bool first = true;
  for (size_t q = 0; q < h->factor.comps.size(); ++q) {
    const double t1 = eval_coef(h->factor.coef_prog[q], mu1, mu_size), t2 = eval_coef(h->factor.coef_prog[q], mu2, mu_size);
    const double ratio = t1 / t2;
    alpha = first ? ratio : std::min(alpha, ratio);
    gamma = first ? ratio : std::max(gamma, ratio);
    first = false;
  }
}

struct IndicatorSums {           // per subdomain (global numbering)
  std::vector<double> s[9];      // sums of rows 0..8 (row 6: minimum)
};

// device part of an estimator evaluation: Oswald vertex means, the per-cell indicator pass and the segmented reductions
// of its nine rows.  Stream ordered, no host synchronisation; u is expected in h->tmp_local (owned part filled in).
void indicators_device(hdd_swipdg* h, const hdd_parameters* prm, bool exchange_halo, int parts = 7) {
  hdd_mesh* m = h->mesh;
  cudaStream_t s = m->stream;
  const int nl = h->nl;
  if (exchange_halo) m->halo_exchange(h->tmp_local.p, nl);
  if (!h->vertex_mean.p) h->vertex_mean.alloc(size_t(m->n_verts_loc));
  if (parts & 1)
    launch_oswald_vertex_means(m->vptr.p, m->vdof.p, m->vboundary.p, m->n_verts_loc, h->tmp_local.p, h->vertex_mean.p, s);

  const int ms = prm ? prm->mu_size : 0;
  const double* mu = prm ? prm->mu : nullptr;
  const double* mu_hat = prm && prm->mu_hat ? prm->mu_hat : mu;
  const double* mu_bar = prm && prm->mu_bar ? prm->mu_bar : mu;
  const double* mu_min = prm && prm->parameter_range_min ? prm->parameter_range_min : mu;
  const double* mu_max = prm && prm->parameter_range_max ? prm->parameter_range_max : mu;
  IndicatorArgs a{};
  a.a_mu = make_combo(h, h->factor, mu, ms);
  a.a_hat = make_combo(h, h->factor, mu_hat, ms);
  a.a_bar = make_combo(h, h->factor, mu_bar, ms);
  a.a_cut = a.a_mu;
  a.a_min = make_combo(h, h->factor, mu_min, ms);
  a.a_max = make_combo(h, h->factor, mu_max, ms);
  if (!h->force.has_affine()) HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET, "the force needs an affine part");
  a.fn_table = h->fn_dev.p;
  a.n_fn = int(h->fn_host.size());
  a.force_idx = h->force.affine.idx;
  a.force_order = h->force.affine.order;
  a.u_local = h->tmp_local.p;
  a.vertex_mean = h->vertex_mean.p;
  a.cell_verts = m->cell_verts.p;
  if (!h->ind_out.p) h->ind_out.alloc(size_t(9) * m->n_own);
  a.out = h->ind_out.p;
  if (parts & 2) launch_indicators(h->view(), a, h->fn_host.data(), h->polorder, s);

  const int n_seg = int(m->seg_sub.size());
  if (!h->seg_out.p) h->seg_out.alloc(size_t(9) * std::max(n_seg, 1));
  if (parts & 4)
    launch_segment_reduce(h->ind_out.p, int64_t(m->n_own), 9, 1u << 6, m->d_seg_ptr.p, n_seg, h->seg_out.p, s);  // row 6: minimum
}

void check_estimator_space(const hdd_swipdg* h) {
  if (h->mesh->kind != HDD_SIMPLEX2D)
    HDD_THROW(HDD_ERR_USING_THIS_WRONG, "the estimators are only available on 2d simplex grids (estimators/swipdg.hh:71)");
  if (h->polorder != 1)
    HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "the estimators need polOrder 1 (Oswald interpolation and RT0 reconstruction, estimators/swipdg.hh:149,359)");
}

// runs the two estimator passes and reduces the per-cell rows per subdomain
void run_indicators(hdd_swipdg* h, const double* u_host, const hdd_parameters* prm, IndicatorSums& sums) {
  hdd_mesh* m = h->mesh;
  cudaStream_t s = m->stream;
  check_estimator_space(h);
  const int nl = h->nl;
  const size_t loc = size_t(m->n_loc) * nl, rows = size_t(h->n_rows);
  if (!h->tmp_local.p) { h->tmp_local.alloc(loc); h->tmp_local.zero(s); }
  if (u_host) {
    HDD_CUDA(h2d_async(h->tmp_local.p + size_t(m->own0) * nl, u_host, rows * sizeof(double), s));
  } else {
    if (!h->have_solution) HDD_THROW(HDD_ERR_USING_THIS_WRONG, "no vector given and no solution available");
    HDD_CUDA(cudaMemcpyAsync(h->tmp_local.p + size_t(m->own0) * nl, h->x.p, rows * sizeof(double), cudaMemcpyDeviceToDevice, s));
  }
  indicators_device(h, prm, true);
  h->estimator_vector_resident = true;
  const int n_seg = int(m->seg_sub.size());
  std::vector<double> seg(size_t(9) * std::max(n_seg, 1));
  HDD_CUDA(cudaMemcpyAsync(seg.data(), h->seg_out.p, seg.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
  HDD_CUDA(cudaStreamSynchronize(s));
  const int ns = m->n_subdomains;
  for (int r = 0; r < 9; ++r) sums.s[r].assign(size_t(ns), r == 6 ? 1e300 : 0.0);
  for (int g = 0; g < n_seg; ++g)
    for (int r = 0; r < 9; ++r) {
      double& dst = sums.s[r][size_t(m->seg_sub[size_t(g)])];
      const double v = seg[size_t(r) * n_seg + g];
      dst = r == 6 ? std::min(dst, v) : dst + v;
    }
  if (m->world > 1) {
    // per-subdomain values live on their owner; make them global (sum of zeros elsewhere / min of +huge)
    DevBuf<double> buf;
    std::vector<double> flat(size_t(9) * ns);
    for (int r = 0; r < 9; ++r) std::copy(sums.s[r].begin(), sums.s[r].end(), flat.begin() + size_t(r) * ns);
    buf.upload(flat.data(), flat.size(), s);
    Nccl& nc = Nccl::get();
    nc.all_reduce_sum(buf.p, size_t(6) * ns, m->comm, s);
    nc.all_reduce_min(buf.p + size_t(6) * ns, size_t(ns), m->comm, s);
    nc.all_reduce_sum(buf.p + size_t(7) * ns, size_t(2) * ns, m->comm, s);
    HDD_CUDA(cudaMemcpyAsync(flat.data(), buf.p, flat.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
    HDD_CUDA(cudaStreamSynchronize(s));
    for (int r = 0; r < 9; ++r) std::copy(flat.begin() + size_t(r) * ns, flat.begin() + size_t(r + 1) * ns, sums.s[r].begin());
  }
}

double total(const std::vector<double>& v) {
  double s = 0.0;
  for (double x : v) s += x;
  return s;
}

const char* const kEstimatorTypes[] = {"eta_NC_ESV2007", "eta_R_ESV2007",  "eta_R_ESV2007_*", "eta_DF_ESV2007", "eta_ESV2007",
                                       "eta_ESV2007_alt", "eta_NC_OS2014", "eta_R_OS2014",    "eta_R_OS2014_*", "eta_DF_OS2014",
                                       "eta_DF_OS2014_*", "eta_OS2014",    "eta_OS2014_*"};

}  // namespace

extern "C" {

int hdd_swipdg_create(hdd_mesh* mesh, int polorder, const hdd_problem* problem, hdd_swipdg** out) {
  return guarded([&] {
    if (!out) HDD_THROW(HDD_ERR_WRONG_INPUT, "out is NULL");
    *out = nullptr;
    if (!mesh || !problem) HDD_THROW(HDD_ERR_WRONG_INPUT, "mesh or problem is NULL");
    if (polorder != 1 && polorder != 2) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "polorder " << polorder << " (p = 1 and p = 2 only)");
    mesh->set_device();
    PhaseTimer pt("hdd_swipdg_create", mesh->stream);
    std::unique_ptr<hdd_swipdg> h(new hdd_swipdg);
    h->mesh = mesh;
    h->polorder = polorder;
    h->nl = n_local_dofs(mesh->kind, polorder);
    if (mesh->n_global * h->nl > int64_t(INT32_MAX)) HDD_THROW(HDD_ERR_WRONG_INPUT, "too many DoFs for 32-bit column indices");
    h->sub_dof_offsets.resize(mesh->sub_cell_offsets.size());
    for (size_t k = 0; k < mesh->sub_cell_offsets.size(); ++k) h->sub_dof_offsets[k] = h->nl * mesh->sub_cell_offsets[k];
    h->parameter_name = problem->parameter_name ? problem->parameter_name : "";
    h->parameter_size = problem->parameter_name ? problem->parameter_size : 0;
    if (h->parameter_size < 0 || h->parameter_size > 4) HDD_THROW(HDD_ERR_WRONG_INPUT, "parameter_size must be in [0,4]");
    h->factor = add_affine(h.get(), problem->diffusion_factor, "diffusion_factor");
    h->force = add_affine(h.get(), problem->force, "force");
    h->dirichlet = add_affine(h.get(), problem->dirichlet, "dirichlet");
    h->neumann = add_affine(h.get(), problem->neumann, "neumann");
    if (!h->factor.parametric() && !h->factor.has_affine())
      HDD_THROW(HDD_ERR_WRONG_INPUT, "The diffusion factor must not be empty!");
    const bool parametric = h->factor.parametric() || h->force.parametric() || h->dirichlet.parametric() || h->neumann.parametric();
    if (parametric && h->parameter_size == 0)
      HDD_THROW(HDD_ERR_WRONG_INPUT, "parametric data functions but no parameter_name / parameter_size given");
    if (problem->diffusion_tensor) {
      h->has_tensor = true;
      if (mesh->whole) {
        h->tensor.upload(problem->diffusion_tensor, size_t(mesh->n_loc) * 4, mesh->stream);
      } else {
        std::vector<double> loc(size_t(mesh->n_loc) * 4);
        for (int32_t lc = 0; lc < mesh->n_loc; ++lc)
          for (int k = 0; k < 4; ++k) loc[size_t(lc) * 4 + k] = problem->diffusion_tensor[int64_t(mesh->gid(lc)) * 4 + k];
        h->tensor.upload(loc.data(), loc.size(), mesh->stream);
        HDD_CUDA(cudaStreamSynchronize(mesh->stream));  // loc dies with this scope
      }
    }
    h->fn_dev.upload(h->fn_host.data(), h->fn_host.size(), mesh->stream);
    HDD_CUDA(cudaStreamSynchronize(mesh->stream));
    h->n_rows = int64_t(mesh->n_own) * h->nl;
    h->nnz = mesh->n_blocks * h->nl * h->nl;

    // affine structure of the system matrix (discretizations/swipdg.hh:228-247) ...
    for (size_t q = 0; q < h->factor.comps.size(); ++q) {
      MatrixPart p;
      p.coef_expr = h->factor.coef_expr[q];
      p.coef_prog = h->factor.coef_prog[q];
      p.factor = h->factor.comps[q];
      h->lhs_comps.push_back(std::move(p));
    }
    if (h->factor.has_affine()) {
      h->lhs_affine.reset(new MatrixPart);
      h->lhs_affine->factor = h->factor.affine;
    }
    // ... and of the rhs (:253-332): force parts, then the (factor part x dirichlet part) products
    const std::string pname = h->parameter_name.empty() ? "mu" : h->parameter_name;
    auto affine_rhs = [&]() -> VectorPart& {
      if (!h->rhs_affine) h->rhs_affine.reset(new VectorPart);
      return *h->rhs_affine;
    };
    for (size_t q = 0; q < h->force.comps.size(); ++q) {
      VectorPart p;
      p.coef_expr = h->force.coef_expr[q];
      p.coef_prog = h->force.coef_prog[q];
      p.terms.push_back({0, h->force.comps[q], FnRef{}});
      h->rhs_comps.push_back(std::move(p));
    }
    if (h->force.has_affine()) affine_rhs().terms.push_back({0, h->force.affine, FnRef{}});
    if (h->factor.has_affine() && h->dirichlet.has_affine())
      affine_rhs().terms.push_back({1, h->factor.affine, h->dirichlet.affine});
    if (h->factor.has_affine())
      for (size_t q = 0; q < h->dirichlet.comps.size(); ++q) {
        VectorPart p;
        p.coef_expr = h->dirichlet.coef_expr[q];
        p.coef_prog = h->dirichlet.coef_prog[q];
        p.terms.push_back({1, h->factor.affine, h->dirichlet.comps[q]});
        h->rhs_comps.push_back(std::move(p));
      }
    if (h->dirichlet.has_affine())
      for (size_t q = 0; q < h->factor.comps.size(); ++q) {
        VectorPart p;
        p.coef_expr = h->factor.coef_expr[q];
        p.coef_prog = h->factor.coef_prog[q];
        p.terms.push_back({1, h->factor.comps[q], h->dirichlet.affine});
        h->rhs_comps.push_back(std::move(p));
      }
    for (size_t pp = 0; pp < h->factor.comps.size(); ++pp)
      for (size_t qq = 0; qq < h->dirichlet.comps.size(); ++qq) {
        VectorPart p;
        p.coef_expr = "(" + h->factor.coef_expr[pp] + ")*(" + h->dirichlet.coef_expr[qq] + ")";
        p.coef_prog = compile_expression(p.coef_expr, pname);
        p.terms.push_back({1, h->factor.comps[pp], h->dirichlet.comps[qq]});
        h->rhs_comps.push_back(std::move(p));
      }
    // ... Neumann parts (:335-356): L2Face on the Neumann intersections
    for (size_t q = 0; q < h->neumann.comps.size(); ++q) {
      VectorPart p;
      p.coef_expr = h->neumann.coef_expr[q];
      p.coef_prog = h->neumann.coef_prog[q];
      p.terms.push_back({2, h->neumann.comps[q], FnRef{}});
      h->rhs_comps.push_back(std::move(p));
    }
    if (h->neumann.has_affine() && !h->neumann.affine.zero) affine_rhs().terms.push_back({2, h->neumann.affine, FnRef{}});
    if (h->lhs_comps.size() + 1 > size_t(kMaxParts) || h->rhs_comps.size() + 1 > size_t(kMaxParts))
      HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "more than " << kMaxParts - 1 << " affine components");
    pt.lap("all");
    *out = h.release();
  });
}

int hdd_swipdg_destroy(hdd_swipdg* h) {
  return guarded([&] {
    if (h) {
      cudaSetDevice(h->mesh->device);
      delete h;
    }
  });
}

int hdd_swipdg_init(hdd_swipdg* h) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    if (h->initialized) return;
    hdd_mesh* m = h->mesh;
    m->set_device();
    cudaStream_t s = m->stream;
    PhaseTimer pt("hdd_swipdg_init", s);
    for (auto& p : h->lhs_comps) p.values.alloc(size_t(h->nnz));
    if (h->lhs_affine) h->lhs_affine->values.alloc(size_t(h->nnz));
    for (auto& p : h->rhs_comps) p.values.alloc(size_t(h->n_rows));
    if (h->rhs_affine) h->rhs_affine->values.alloc(size_t(h->n_rows));
    pt.lap("allocate");
    assemble_all(h);
    assemble_products(h);
    HDD_CUDA(cudaStreamSynchronize(s));
    pt.lap("assemble");
    h->initialized = true;
  });
}

int hdd_swipdg_assemble(hdd_swipdg* h, double* seconds) {
  return guarded([&] {
    require_init(h);
    hdd_mesh* m = h->mesh;
    m->set_device();
    cudaEvent_t e0, e1;
    HDD_CUDA(cudaEventCreate(&e0));
    HDD_CUDA(cudaEventCreate(&e1));
    HDD_CUDA(cudaEventRecord(e0, m->stream));
    assemble_all(h);
    HDD_CUDA(cudaEventRecord(e1, m->stream));
    HDD_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    HDD_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (seconds) *seconds = double(ms) * 1e-3;
  });
}

int hdd_num_dofs(const hdd_swipdg* h, int64_t* n_global, int64_t* n_owned) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    if (n_global) *n_global = h->mesh->n_global * h->nl;
    if (n_owned) *n_owned = h->n_rows;
  });
}

int hdd_pattern(hdd_swipdg* h, int64_t* n_rows, int64_t* nnz, const int64_t** rowptr_dev, const int32_t** col_dev) {
  return guarded([&] {
    require_init(h);
    if (n_rows) *n_rows = h->n_rows;
    if (nnz) *nnz = h->nnz;
    // K1 part 2: the expanded CSR index arrays.  The pattern itself - which blocks a row of cells has, in sorted order - is
    // the block-offset array built with the mesh (K1 part 1) together with the neighbour table; every kernel works on that
    // block-compressed form and never reads an index.  The 12 bytes per non-zero of rowptr / col (5.9 GB at 4096^2 Q1, 3.1 ms
    // to write) are a view for consumers of the matrix and are materialised when the first one asks for them.
    if ((rowptr_dev || col_dev) && !h->rowptr.p) {
      hdd_mesh* m = h->mesh;
      m->set_device();
      h->rowptr.alloc(size_t(h->n_rows) + 1);
      h->col.alloc(size_t(h->nnz));
      if (h->n_rows == 0) HDD_CUDA(cudaMemsetAsync(h->rowptr.p, 0, sizeof(int64_t), m->stream));
      launch_fill_csr(h->view(), h->rowptr.p, h->col.p, m->stream);
      HDD_CUDA(cudaStreamSynchronize(m->stream));
    }
    if (rowptr_dev) *rowptr_dev = h->rowptr.p;
    if (col_dev) *col_dev = h->col.p;
  });
}

int hdd_num_components(const hdd_swipdg* h, int which, int* n_components, int* has_affine_part) {
  return guarded([&] {
    require_init(h);
    if (which != HDD_LHS && which != HDD_RHS) HDD_THROW(HDD_ERR_WRONG_INPUT, "which must be HDD_LHS or HDD_RHS");
    if (n_components) *n_components = int(which == HDD_LHS ? h->lhs_comps.size() : h->rhs_comps.size());
    if (has_affine_part) *has_affine_part = (which == HDD_LHS ? bool(h->lhs_affine) : bool(h->rhs_affine)) ? 1 : 0;
  });
}

int hdd_component_values(hdd_swipdg* h, int which, int q, const double** values_dev, int64_t* count) {
  return guarded([&] {
    require_init(h);
    if (which != HDD_LHS && which != HDD_RHS) HDD_THROW(HDD_ERR_WRONG_INPUT, "which must be HDD_LHS or HDD_RHS");
    const double* p = nullptr;
    if (which == HDD_LHS) {
      if (q == -1) {
        if (!h->lhs_affine) HDD_THROW(HDD_ERR_USING_THIS_WRONG, "the system matrix has no affine part");
        p = h->lhs_affine->values.p;
      } else {
        if (q < 0 || q >= int(h->lhs_comps.size())) HDD_THROW(HDD_ERR_INDEX_OUT_OF_RANGE, "component " << q);
        p = h->lhs_comps[size_t(q)].values.p;
      }
      if (count) *count = h->nnz;
    } else {
      if (q == -1) {
        if (!h->rhs_affine) HDD_THROW(HDD_ERR_USING_THIS_WRONG, "the rhs has no affine part");
        p = h->rhs_affine->values.p;
      } else {
        if (q < 0 || q >= int(h->rhs_comps.size())) HDD_THROW(HDD_ERR_INDEX_OUT_OF_RANGE, "component " << q);
        p = h->rhs_comps[size_t(q)].values.p;
      }
      if (count) *count = h->n_rows;
    }
    if (values_dev) *values_dev = p;
  });
}

int hdd_component_coefficient(const hdd_swipdg* h, int which, int q, const char** expression) {
  return guarded([&] {
    require_init(h);
    if (which != HDD_LHS && which != HDD_RHS) HDD_THROW(HDD_ERR_WRONG_INPUT, "which must be HDD_LHS or HDD_RHS");
    const size_t n = which == HDD_LHS ? h->lhs_comps.size() : h->rhs_comps.size();
    if (q < 0 || size_t(q) >= n) HDD_THROW(HDD_ERR_INDEX_OUT_OF_RANGE, "component " << q);
    if (expression)
      *expression = which == HDD_LHS ? h->lhs_comps[size_t(q)].coef_expr.c_str() : h->rhs_comps[size_t(q)].coef_expr.c_str();
  });
}

int hdd_evaluate_coefficients(const hdd_swipdg* h, int which, const double* mu, int mu_size, double* theta) {
  return guarded([&] {
    require_init(h);
    check_mu(h, mu, mu_size, "mu");
    if (which == HDD_LHS)
      for (size_t q = 0; q < h->lhs_comps.size(); ++q) theta[q] = eval_coef(h->lhs_comps[q].coef_prog, mu, mu_size);
    else if (which == HDD_RHS)
      for (size_t q = 0; q < h->rhs_comps.size(); ++q) theta[q] = eval_coef(h->rhs_comps[q].coef_prog, mu, mu_size);
    else
      HDD_THROW(HDD_ERR_WRONG_INPUT, "which must be HDD_LHS or HDD_RHS");
  });
}

int hdd_copy_to_host(hdd_swipdg* h, void* dst_host, const void* src_dev, size_t bytes) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    h->mesh->set_device();
    HDD_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, h->mesh->stream));
    HDD_CUDA(cudaStreamSynchronize(h->mesh->stream));
  });
}

int hdd_sync(hdd_swipdg* h) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    h->mesh->set_device();
    HDD_CUDA(cudaStreamSynchronize(h->mesh->stream));
  });
}

int hdd_apply(hdd_swipdg* h, const double* mu, int mu_size, const double* x_host, double* y_host) {
  return guarded([&] {
    require_init(h);
    check_mu(h, mu, mu_size, "mu");
    hdd_mesh* m = h->mesh;
    m->set_device();
    cudaStream_t s = m->stream;
    const double* vals = freeze_lhs(h, mu, mu_size);
    const size_t loc = size_t(m->n_loc) * h->nl, rows = size_t(h->n_rows);
    if (!h->tmp_local.p) { h->tmp_local.alloc(loc); h->tmp_local.zero(s); }
    DevBuf<double> y;
    y.alloc(rows);
    HDD_CUDA(h2d_async(h->tmp_local.p + size_t(m->own0) * h->nl, x_host, rows * sizeof(double), s));
    m->halo_exchange(h->tmp_local.p, h->nl);
    launch_spmv(h->view(), vals, h->tmp_local.p, y.p, s);
    HDD_CUDA(cudaMemcpyAsync(y_host, y.p, rows * sizeof(double), cudaMemcpyDeviceToHost, s));
    HDD_CUDA(cudaStreamSynchronize(s));
  });
}

int hdd_residual(hdd_swipdg* h, const double* mu, int mu_size, double* relative_residual, double* fp64_floor) {
  return guarded([&] {
    require_init(h);
    check_mu(h, mu, mu_size, "mu");
    if (!h->have_solution) HDD_THROW(HDD_ERR_USING_THIS_WRONG, "no solution available, call hdd_solve first");
    hdd_mesh* m = h->mesh;
    if (m->purely_neumann) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "hdd_residual for the modified pure-Neumann system");
    m->set_device();
    cudaStream_t s = m->stream;
    const double* vals = freeze_lhs(h, mu, mu_size);
    freeze_rhs(h, mu, mu_size);
    const size_t loc = size_t(m->n_loc) * h->nl, rows = size_t(h->n_rows);
    if (!h->tmp_local.p) { h->tmp_local.alloc(loc); h->tmp_local.zero(s); }
    HDD_CUDA(cudaMemcpyAsync(h->tmp_local.p + size_t(m->own0) * h->nl, h->x.p, rows * sizeof(double), cudaMemcpyDeviceToDevice, s));
    m->halo_exchange(h->tmp_local.p, h->nl);
    launch_spmv(h->view(), vals, h->tmp_local.p, h->q.p, s);
    launch_residual_norms(h->b.p, h->q.p, h->x.p, int64_t(rows), vals, h->nnz, h->partial.p, h->sc.p, s);
    if (m->world > 1) {
      Nccl::get().all_reduce_sum(&h->sc.p->red[0], 3, m->comm, s);
      // max |A_ij| over the ranks: -min(-v)
      DevBuf<double> neg;
      double amax_local = 0.0;
      HDD_CUDA(cudaMemcpyAsync(&amax_local, &h->sc.p->red[3], sizeof(double), cudaMemcpyDeviceToHost, s));
      HDD_CUDA(cudaStreamSynchronize(s));
      amax_local = -amax_local;
      neg.upload(&amax_local, 1, s);
      Nccl::get().all_reduce_min(neg.p, 1, m->comm, s);
      HDD_CUDA(cudaMemcpyAsync(&amax_local, neg.p, sizeof(double), cudaMemcpyDeviceToHost, s));
      HDD_CUDA(cudaStreamSynchronize(s));
      amax_local = -amax_local;
      HDD_CUDA(h2d_async(&h->sc.p->red[3], &amax_local, sizeof(double), s));
      HDD_CUDA(cudaStreamSynchronize(s));
    }
    double red[4] = {0.0, 0.0, 0.0, 0.0};
    HDD_CUDA(cudaMemcpyAsync(red, &h->sc.p->red[0], sizeof(red), cudaMemcpyDeviceToHost, s));
    HDD_CUDA(cudaStreamSynchronize(s));
    if (relative_residual) *relative_residual = red[1] > 0.0 ? std::sqrt(red[0] / red[1]) : std::sqrt(red[0]);
    // what b - A x can resolve in fp64: one SpMV row sums (1 + n_faces) n_loc products of size <= max|A| |x|
    if (fp64_floor)
      *fp64_floor = red[1] > 0.0 ? 1.1102230246251565e-16 * double((m->nf + 1) * h->nl) * red[3] * std::sqrt(red[2] / red[1]) : 0.0;
  });
}

int hdd_solver_types(const char* const** types, int* n_types) {
  return guarded([&] {
    static const std::vector<const char*> names = [] {
      std::vector<const char*> v;
      for (const SolverTypeName& e : kSolverTypes) v.push_back(e.name);
      return v;
    }();
    if (types) *types = names.data();
    if (n_types) *n_types = int(names.size());
  });
}

namespace {

struct CgStart {
  const double* vals = nullptr;  // the frozen operator the iteration reads
  bool p2p = false;
  const PeerView* peer = nullptr;
};

// The start of a CG solve, shared by hdd_solve and hdd_precondition: A(mu) frozen (and b(mu) into c.b if freeze_b), the
// pure-Neumann fix, the preconditioner's set-up, the peer-memory decision, then x = 0, r = b, p = z = M^-1 b and
// rz[0] = r.z.  The caller provides c.b, c.x, c.r, c.z (block Jacobi and multigrid), c.p, c.q, c.partial and c.sc.
CgStart start_cg(hdd_swipdg* h, SolverType type, const double* mu, int mu_size, bool freeze_b, double precision, int max_iter,
                 CgBuffers& c) {
  hdd_mesh* m = h->mesh;
  cudaStream_t s = m->stream;
  SolvePhases& pt = phase_timer();
  CgStart st;
  const double* vals = freeze_lhs(h, mu, mu_size);
  if (freeze_b) freeze_rhs(h, mu, mu_size);
  pt.mark("setup: freeze", s);
  const MeshView v = h->view();
  if (m->purely_neumann) {
    // discretizations/base.hh:337-345: unit_row(0), rhs[0] = 0, solve, subtract the mean
    if (m->world > 1) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "pure Neumann problems on more than one GPU");
    if (!h->frozen.p) h->frozen.alloc(size_t(h->nnz));
    if (vals != h->frozen.p)
      HDD_CUDA(cudaMemcpyAsync(h->frozen.p, vals, size_t(h->nnz) * sizeof(double), cudaMemcpyDeviceToDevice, s));
    launch_unit_row_col0(v, h->frozen.p, h->b.p, s);  // c.b is h->b here: hdd_precondition refuses this case
    vals = h->frozen.p;
  }
  c.values = vals;
  c.dinv = h->dinv.p;
  if (uses_block_inverses(type)) {
    if (!h->dinv_block.p) h->dinv_block.alloc(size_t(m->n_own) * h->nl * h->nl);
    launch_invert_diag_blocks(v, vals, h->dinv_block.p, s);
    pt.mark("setup: block inverses", s);
    c.dinv_block = h->dinv_block.p;
    if (is_multigrid(type)) mg_setup(h, vals, type);
  } else {
    c.z = nullptr;
    launch_extract_dinv(v, vals, type == SolverType::diagonal, h->dinv.p, s);
  }
  Nccl& nc = Nccl::get();
  const bool multi = m->world > 1;
  // multi GPU, Q1, Jacobi / identity: fused SpMV + halo read over peer memory instead of pack + send/recv
  bool p2p = multi && p2p_wanted() && !uses_block_inverses(type) && cg_spmv_uses_tma(v);
  if (multi && !uses_block_inverses(type)) {  // the decision must be collective: a rank without owned cells large enough would disagree
    DevBuf<double> vote;
    double want = p2p ? 0.0 : 1.0;
    vote.upload(&want, 1, s);
    nc.all_reduce_sum(vote.p, 1, m->comm, s);
    HDD_CUDA(cudaMemcpyAsync(&want, vote.p, sizeof(double), cudaMemcpyDeviceToHost, s));
    HDD_CUDA(cudaStreamSynchronize(s));
    p2p = (want == 0.0);
  }
  if (p2p) p2p = setup_p2p(h);
  pt.mark("setup: solver vote", s);
  if (p2p) {
    // Jacobi diagonal including the halo (static during the solve): owned part computed here, halo exchanged once
    double* dl = h->dinv_local.p;
    HDD_CUDA(cudaMemcpyAsync(dl + size_t(m->own0) * h->nl, h->dinv.p, size_t(h->n_rows) * sizeof(double), cudaMemcpyDeviceToDevice, s));
    m->halo_exchange(dl, h->nl);
    c.p_alt = h->p_alt.p;
    st.peer = &h->peer_view;
  }
  launch_cg_init(v, c, precision, max_iter, s);
  if (is_multigrid(type)) mg_apply(h, nullptr, c.r, c.z, c.p + size_t(m->own0) * h->nl, c.partial, c.sc);
  if (multi) nc.all_reduce_sum(&c.sc->red[1], 2, m->comm, s);
  launch_cg_init_finish(v, c, s);
  pt.mark("setup: cg init", s);
  st.vals = vals;
  st.p2p = p2p;
  return st;
}

}  // namespace

int hdd_solve(hdd_swipdg* h, const char* type, double precision, int max_iter, const double* mu, int mu_size,
              double* x_host, hdd_solve_info* info) {
  return guarded([&] {
    require_init(h);
    check_mu(h, mu, mu_size, "mu");
    const SolverType solver = parse_solver_type(type);
    if (!(precision > 0.0)) HDD_THROW(HDD_ERR_WRONG_INPUT, "precision must be positive");
    hdd_mesh* m = h->mesh;
    m->set_device();
    cudaStream_t s = m->stream;
    ensure_solve_workspace(h);
    if (uses_block_inverses(solver) && !h->z.p) h->z.alloc(size_t(h->n_rows));
    cudaEvent_t e0, e1;
    HDD_CUDA(cudaEventCreate(&e0));
    HDD_CUDA(cudaEventCreate(&e1));
    HDD_CUDA(cudaEventRecord(e0, s));
    SolvePhases& pt = phase_timer();
    pt.begin(s);
    h->last_type = solver;
    CgBuffers c{};
    c.b = h->b.p;
    c.x = h->x.p;
    c.r = h->r.p;
    c.z = h->z.p;
    c.p = h->p.p;
    c.q = h->q.p;
    c.partial = h->partial.p;
    c.sc = h->sc.p;
    if (!c.b) {  // freeze_rhs allocates b at the first solve
      h->b.alloc(size_t(h->n_rows));
      c.b = h->b.p;
    }
    const CgStart st = start_cg(h, solver, mu, mu_size, true, precision, max_iter, c);
    const double* vals = st.vals;
    const bool p2p = st.p2p;
    const PeerView* peer = st.peer;
    const MeshView v = h->view();
    Nccl& nc = Nccl::get();
    const bool multi = m->world > 1;
    // One CG iteration = 3 kernels (+ 2 all-reduces, + ~100 small multigrid kernels for cg.mg / cg.mg2 / cg.mg2.simplex).  The first batch is
    // launched directly (one-time attribute / buffer set-up happens there); after that two iterations (parity 0 and 1)
    // are captured into a CUDA graph and replayed, so a launch-bound iteration costs one graph launch instead of up to
    // a hundred kernel launches and does not stall the GPU when the host thread is delayed.  HDD_CG_GRAPH=0 disables it.
    auto iteration = [&](int parity) {
      if (multi && !p2p) { m->halo_exchange(c.p, h->nl); pt.mark("halo exchange (p)", s); }
      launch_cg_spmv(v, c, parity, s, peer);
      pt.mark("spmv", s);
      if (multi) { nc.all_reduce_sum(&c.sc->red[0], 1, m->comm, s); pt.mark("all-reduce p.q", s); }
      launch_cg_update(v, c, parity, s);
      pt.mark("update", s);
      if (is_multigrid(solver)) mg_apply(h, &c.sc->done[parity], c.r, c.z, nullptr, c.partial, c.sc);
      if (multi) { nc.all_reduce_sum(&c.sc->red[1], 2, m->comm, s); pt.mark("all-reduce r.z", s); }
      launch_cg_direction(v, c, parity, s);
      pt.mark("direction", s);
    };
    static const bool graphs_wanted = [] {
      const char* e = std::getenv("HDD_CG_GRAPH");
      return !(e && e[0] == '0') && !phase_timer().on;
    }();
    hdd_swipdg::CgGraph& cached = h->cg_graph[int(solver)];
    const void* key[5] = {vals, c.p_alt, peer, c.dinv_block, m->send_buf.p};
    if (cached.exec && std::memcmp(cached.key, key, sizeof(key)) != 0) {
      cudaGraphExecDestroy(cached.exec);
      cached.exec = nullptr;
    }
    bool capture_failed = false;
    double rr_prev = 1e300;
    int par = 0, launched = 0, batch = is_multigrid(solver) ? 8 : 16;
    bool first_batch = !cached.exec;  // a cached graph means every one-time set-up has already happened
    for (;;) {
      if (!first_batch && graphs_wanted && !cached.exec && !capture_failed) {
        const int64_t before = hdd_kernel_launches();
        cudaGraph_t g = nullptr;
        bool ok = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
        if (ok) {
          try {
            iteration(0);
            iteration(1);
          } catch (const Error&) {
            ok = false;
          }
          if (cudaStreamEndCapture(s, &g) != cudaSuccess || !g) ok = false;
          if (ok && cudaGraphInstantiate(&cached.exec, g, 0) != cudaSuccess) ok = false;
          if (g) cudaGraphDestroy(g);
        }
        cached.launches = hdd_kernel_launches() - before;
        g_kernel_launches.fetch_sub(cached.launches);  // captured, not launched yet
        if (ok) {
          std::memcpy(cached.key, key, sizeof(key));
        } else {
          cudaGetLastError();
          if (cached.exec) cudaGraphExecDestroy(cached.exec);
          cached.exec = nullptr;
          capture_failed = true;
        }
      }
      if (cached.exec && graphs_wanted) {
        for (int k = 0; k < batch; k += 2) HDD_CUDA(cudaGraphLaunch(cached.exec, s));
        count_launch(int(cached.launches) * (batch / 2));
        launched += batch;  // batch is even: the parity is back at its value from the start of the batch
      } else {
        for (int k = 0; k < batch; ++k) {
          iteration(par);
          par ^= 1;
          ++launched;
        }
      }
      first_batch = false;
      HDD_CUDA(cudaMemcpyAsync(h->sc_host, h->sc.p, sizeof(CgScalars), cudaMemcpyDeviceToHost, s));
      HDD_CUDA(cudaStreamSynchronize(s));
      if (h->sc_host->done[par]) break;
      if (launched > max_iter + batch) break;  // cannot happen: done latches at max_it
      // next batch: the iterations still needed at the convergence rate seen so far (iterations launched after
      // convergence are no-ops, but they still cost their launch), at most twice the last batch and at most 256
      {
        const double rr = h->sc_host->rr, target = h->sc_host->tol2 * h->sc_host->bb;
        int next = 2 * batch;
        if (rr > 0.0 && rr < rr_prev && target > 0.0 && rr > target) {
          const double per_it = std::log(rr / rr_prev) / batch;  // < 0
          const double need = std::log(target / rr) / per_it;
          if (need < double(next)) next = int(need) + 1;
        }
        rr_prev = rr;
        batch = std::max(2, std::min(256, (next + 1) & ~1));
      }
    }
    if (m->purely_neumann) launch_subtract_mean(h->x.p, h->n_rows, h->partial.p, h->sc.p, s);
    pt.report(m->rank, launched);
    HDD_CUDA(cudaEventRecord(e1, s));
    HDD_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    HDD_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    h->have_solution = true;
    const CgScalars& sc = *h->sc_host;
    const double relres = sc.bb > 0.0 ? std::sqrt(sc.rr / sc.bb) : 0.0;
    const bool converged = sc.bb == 0.0 || sc.rr <= sc.tol2 * sc.bb;
    if (info) {
      info->iterations = sc.it[par];
      info->converged = converged ? 1 : 0;
      info->relative_residual = relres;
      info->seconds = double(ms) * 1e-3;
      info->seconds_per_iteration = sc.it[par] > 0 ? double(ms) * 1e-3 / sc.it[par] : 0.0;
      info->peer_memory = p2p ? 1 : 0;
    }
    if (x_host) {
      HDD_CUDA(cudaMemcpyAsync(x_host, h->x.p, size_t(h->n_rows) * sizeof(double), cudaMemcpyDeviceToHost, s));
      HDD_CUDA(cudaStreamSynchronize(s));
    }
    if (!converged)
      HDD_THROW(HDD_ERR_NOT_CONVERGED, "CG did not reach precision " << precision << " in " << sc.it[par]
                                                                     << " iterations (relative residual " << relres << ")");
  });
}

int hdd_precondition(hdd_swipdg* h, const char* type, const double* mu, int mu_size, const double* r_host,
                     double* z_host, double* rz, double* vertex_host) {
  return guarded([&] {
    require_init(h);
    check_mu(h, mu, mu_size, "mu");
    const SolverType solver = parse_solver_type(type);
    if (!r_host || !z_host) HDD_THROW(HDD_ERR_WRONG_INPUT, "r_host and z_host must not be NULL");
    if (vertex_host && !is_multigrid(solver)) HDD_THROW(HDD_ERR_WRONG_INPUT, "vertex_host needs a multigrid solver type");
    hdd_mesh* m = h->mesh;
    if (m->world > 1) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "hdd_precondition on more than one GPU");
    if (m->purely_neumann) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "hdd_precondition for the modified pure-Neumann system");
    m->set_device();
    cudaStream_t s = m->stream;
    ensure_solve_workspace(h);
    const size_t rows = size_t(h->n_rows);
    // scratch copies of everything the set-up writes besides the preconditioner's own state
    DevBuf<double> b, x, r, z, p, q, partial;
    DevBuf<CgScalars> sc;
    b.alloc(rows);
    x.alloc(rows);
    r.alloc(rows);
    z.alloc(rows);
    p.alloc(size_t(m->n_loc) * h->nl);
    q.alloc(rows);
    partial.alloc(size_t(cg_partial_capacity()));
    sc.alloc(1);
    HDD_CUDA(h2d_async(b.p, r_host, rows * sizeof(double), s));
    CgBuffers c{};
    c.b = b.p;
    c.x = x.p;
    c.r = r.p;
    c.z = z.p;
    c.p = p.p;
    c.q = q.p;
    c.partial = partial.p;
    c.sc = sc.p;
    start_cg(h, solver, mu, mu_size, false, 1.0, 1, c);
    HDD_CUDA(cudaMemcpyAsync(z_host, p.p + size_t(m->own0) * h->nl, rows * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (rz) HDD_CUDA(cudaMemcpyAsync(rz, &sc.p->rz[0], sizeof(double), cudaMemcpyDeviceToHost, s));
    if (vertex_host) mg_vertex_result(h, vertex_host);
    HDD_CUDA(cudaStreamSynchronize(s));
  });
}

int hdd_solution_dev(hdd_swipdg* h, const double** x_dev) {
  return guarded([&] {
    require_init(h);
    if (!h->have_solution) HDD_THROW(HDD_ERR_USING_THIS_WRONG, "no solution available, call hdd_solve first");
    if (x_dev) *x_dev = h->x.p;
  });
}

// ---- BlockSWIPDG views ---------------------------------------------------------------------------------------
int hdd_num_subdomains(const hdd_swipdg* h, int* n) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    if (n) *n = h->mesh->n_subdomains;
  });
}

int hdd_subdomain_offsets(const hdd_swipdg* h, const int64_t** offsets_host) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    if (offsets_host) *offsets_host = h->sub_dof_offsets.data();
  });
}

int hdd_neighbouring_subdomains(const hdd_swipdg* h, int ss, const int32_t** neighbours_host, int* n) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    if (ss < 0 || ss >= h->mesh->n_subdomains)
      HDD_THROW(HDD_ERR_INDEX_OUT_OF_RANGE, "0 <= ss < num_subdomains() = " << h->mesh->n_subdomains << " is not true for ss = " << ss << "!");
    const auto& v = h->mesh->sub_neighbours[size_t(ss)];
    if (neighbours_host) *neighbours_host = v.data();
    if (n) *n = int(v.size());
  });
}

int hdd_block_extract(hdd_swipdg* h, int ss, int nn, int q, hdd_csr* out) {
  return guarded([&] {
    require_init(h);
    if (!out) HDD_THROW(HDD_ERR_WRONG_INPUT, "out is NULL");
    std::memset(out, 0, sizeof(*out));
    hdd_mesh* m = h->mesh;
    const int ns = m->n_subdomains, nl = h->nl, nf = m->nf;
    if (ss < 0 || ss >= ns) HDD_THROW(HDD_ERR_INDEX_OUT_OF_RANGE, "0 <= ss < num_subdomains() = " << ns << " is not true for ss = " << ss << "!");
    if (nn < 0 || nn >= ns) HDD_THROW(HDD_ERR_INDEX_OUT_OF_RANGE, "0 <= nn < num_subdomains() = " << ns << " is not true for nn = " << nn << "!");
    if (nn != ss) {
      const auto& nb = m->sub_neighbours[size_t(ss)];
      if (!std::binary_search(nb.begin(), nb.end(), nn))
        HDD_THROW(HDD_ERR_WRONG_INPUT, "Subdomain " << nn << " is not a neighbour of subdomain " << ss
                                                    << " (call neighbouring_subdomains(" << ss << ") to find out)!");
    }
    if (ss < m->sub_first || ss >= m->sub_last) HDD_THROW(HDD_ERR_WRONG_INPUT, "subdomain " << ss << " is not owned by this rank");
    const double* vals_dev = nullptr;
    if (q == -1) {
      if (!h->lhs_affine) HDD_THROW(HDD_ERR_USING_THIS_WRONG, "the system matrix has no affine part");
      vals_dev = h->lhs_affine->values.p;
    } else {
      if (q < 0 || q >= int(h->lhs_comps.size())) HDD_THROW(HDD_ERR_INDEX_OUT_OF_RANGE, "component " << q);
      vals_dev = h->lhs_comps[size_t(q)].values.p;
    }
    m->set_device();
    const int64_t k0 = m->sub_cell_offsets[size_t(ss)] - m->cell_begin, k1 = m->sub_cell_offsets[size_t(ss) + 1] - m->cell_begin;
    std::vector<int64_t> bs(size_t(k1 - k0) + 1);
    HDD_CUDA(cudaMemcpyAsync(bs.data(), m->blk_start.p + k0, bs.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, m->stream));
    HDD_CUDA(cudaStreamSynchronize(m->stream));
    const int64_t v0 = bs.front() * nl * nl, v1 = bs.back() * nl * nl;
    std::vector<double> vals(size_t(v1 - v0));
    HDD_CUDA(cudaMemcpyAsync(vals.data(), vals_dev + v0, vals.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
    HDD_CUDA(cudaStreamSynchronize(m->stream));
    std::vector<int32_t> nbr(size_t(k1 - k0) * nf);  // local neighbour ids of the subdomain's cells
    HDD_CUDA(cudaMemcpyAsync(nbr.data(), m->neigh.p + k0 * nf, nbr.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
    HDD_CUDA(cudaStreamSynchronize(m->stream));
    const int64_t col0 = m->sub_cell_offsets[size_t(nn)], col1 = m->sub_cell_offsets[size_t(nn) + 1];
    out->n_rows = (k1 - k0) * nl;
    out->n_cols = (m->sub_cell_offsets[size_t(nn) + 1] - col0) * nl;
    std::vector<int64_t> rowptr(size_t(out->n_rows) + 1, 0);
    std::vector<int32_t> col;
    std::vector<double> val;
    for (int64_t k = k0; k < k1; ++k) {
      const int32_t self = int32_t(m->own0 + k);
      int32_t cells[5];
      int nb = 0;
      cells[nb++] = self;
      for (int f = 0; f < nf; ++f)
        if (nbr[size_t(k - k0) * nf + f] >= 0) cells[nb++] = nbr[size_t(k - k0) * nf + f];
      std::sort(cells, cells + nb);
      const int64_t base = bs[size_t(k - k0)] * nl * nl - v0;
      for (int i = 0; i < nl; ++i) {
        for (int b = 0; b < nb; ++b) {
          const int64_t gc = m->gid(cells[b]);
          if (gc < col0 || gc >= col1) continue;  // not a cell of subdomain nn
          for (int j = 0; j < nl; ++j) {
            col.push_back(int32_t((gc - col0) * nl + j));
            val.push_back(vals[size_t(base + int64_t(i) * nb * nl + b * nl + j)]);
          }
        }
        rowptr[size_t((k - k0) * nl + i) + 1] = int64_t(col.size());
      }
    }
    out->nnz = int64_t(col.size());
    out->rowptr = static_cast<int64_t*>(std::malloc(rowptr.size() * sizeof(int64_t)));
    out->col = static_cast<int32_t*>(std::malloc(std::max<size_t>(col.size(), 1) * sizeof(int32_t)));
    out->val = static_cast<double*>(std::malloc(std::max<size_t>(val.size(), 1) * sizeof(double)));
    if (!out->rowptr || !out->col || !out->val) throw std::bad_alloc();
    std::memcpy(out->rowptr, rowptr.data(), rowptr.size() * sizeof(int64_t));
    if (!col.empty()) std::memcpy(out->col, col.data(), col.size() * sizeof(int32_t));
    if (!val.empty()) std::memcpy(out->val, val.data(), val.size() * sizeof(double));
  });
}

int hdd_csr_free(hdd_csr* mcsr) {
  return guarded([&] {
    if (!mcsr) return;
    std::free(mcsr->rowptr);
    std::free(mcsr->col);
    std::free(mcsr->val);
    std::memset(mcsr, 0, sizeof(*mcsr));
  });
}

// ---- estimators -------------------------------------------------------------------------------------------------
int hdd_estimators_available(const hdd_swipdg* h, const char* const** types, int* n_types) {
  return guarded([&] {
    if (!h) HDD_THROW(HDD_ERR_WRONG_INPUT, "discretization handle is NULL");
    const bool ok = h->mesh->kind == HDD_SIMPLEX2D;  // specialised for ALUGrid<2,2,simplex,conforming> only
    if (types) *types = kEstimatorTypes;
    if (n_types) *n_types = ok ? 13 : 0;
  });
}

int hdd_indicators(hdd_swipdg* h, const double* u_host, const hdd_parameters* prm, double* out_host) {
  return guarded([&] {
    require_init(h);
    h->mesh->set_device();
    if (h->factor.parametric() && (!prm || !prm->mu)) HDD_THROW(HDD_ERR_WRONG_INPUT, "Given parameters are missing 'mu'!");
    if (prm && prm->mu) check_mu(h, prm->mu, prm->mu_size, "mu");
    IndicatorSums sums;
    run_indicators(h, u_host, prm, sums);
    if (out_host) {
      HDD_CUDA(cudaMemcpyAsync(out_host, h->ind_out.p, size_t(8) * h->mesh->n_own * sizeof(double), cudaMemcpyDeviceToHost,
                               h->mesh->stream));
      HDD_CUDA(cudaStreamSynchronize(h->mesh->stream));
    }
  });
}

int hdd_estimate(hdd_swipdg* h, const char* type_c, const double* u_host, const hdd_parameters* prm, double* eta,
                 double* local_host) {
  return guarded([&] {
    require_init(h);
    hdd_mesh* m = h->mesh;
    m->set_device();
    const std::string type = type_c ? type_c : "";
    int which = -1;
    for (int k = 0; k < 13; ++k)
      if (type == kEstimatorTypes[k]) which = k;
    if (which < 0 || m->kind != HDD_SIMPLEX2D)
      HDD_THROW(HDD_ERR_USING_THIS_WRONG, "Requested type '" << type << "' is not one of available()!");
    const bool esv = which <= 5;
    const bool parametric = h->factor.parametric();
    const int ms = prm ? prm->mu_size : 0;
    // parameter checks in the order of the reference (estimators/block-swipdg.hh:756-773, swipdg.hh:117-118,552-555)
    if (h->force.parametric()) HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET, "Not implemented for parametric force!");
    if (h->dirichlet.parametric()) HDD_THROW(HDD_ERR_REQUIREMENTS_NOT_MET, "Not implemented for parametric dirichlet!");
    if (parametric) {
      auto need = [&](const double* p, const char* key) {
        if (!prm || !p) HDD_THROW(HDD_ERR_WRONG_INPUT, "Given parameters are missing '" << key << "'!");
        check_mu(h, p, ms, key);
      };
      const bool os_full = which == 11 || which == 12;
      if (which == 1) HDD_THROW(HDD_ERR_NOT_IMPLEMENTED, "Not implemented yet for parametric problems!");  // swipdg.hh:241-242
      if (which == 0 || which == 6 || os_full || which == 4 || which == 5) need(prm ? prm->mu_bar : nullptr, "mu_bar");
      if (which == 2 || which == 3 || which == 8 || which == 9 || which == 10 || os_full || which == 4 || which == 5)
        need(prm ? prm->mu : nullptr, "mu");
      if (which == 3 || which == 9 || which == 10 || os_full || which == 4 || which == 5) need(prm ? prm->mu_hat : nullptr, "mu_hat");
      if (which == 7 || which == 8 || os_full) {
        need(prm ? prm->parameter_range_min : nullptr, "parameter_range_min");
        need(prm ? prm->parameter_range_max : nullptr, "parameter_range_max");
      }
    }
    // the kernels need *some* mu to freeze the factor with even if this type does not use it
    hdd_parameters eff{};
    if (prm) eff = *prm;
    if (parametric) {
      const double* any = eff.mu ? eff.mu : eff.mu_bar ? eff.mu_bar : eff.mu_hat ? eff.mu_hat : eff.parameter_range_min;
      if (!eff.mu) eff.mu = any;
    }
    IndicatorSums S;
    run_indicators(h, u_host, parametric ? &eff : prm, S);
    const int ns = m->n_subdomains;
    const double cp = 1.0 / (kPi * kPi);
    // OS2014 residuals: per subdomain C_P diam(S)^2 / c_S * sum_T int (f - ...)^2  (estimators/block-swipdg.hh:288-309)
    std::vector<double> r_os, rstar_os;
    r_os.assign(size_t(ns), 0.0);
    rstar_os.assign(size_t(ns), 0.0);
    for (int sdm = 0; sdm < ns; ++sdm) {
      const double w = cp * m->sub_diameter[size_t(sdm)] * m->sub_diameter[size_t(sdm)] / S.s[6][size_t(sdm)];
      r_os[size_t(sdm)] = w * S.s[1][size_t(sdm)];
      rstar_os[size_t(sdm)] = w * S.s[7][size_t(sdm)];
    }
    double a_bar = 1, g_bar = 1, a_hat = 1, g_hat = 1;
    if (parametric && (which == 11 || which == 12)) {
      alpha_gamma(h, prm->mu, prm->mu_bar, ms, a_bar, g_bar);
      alpha_gamma(h, prm->mu, prm->mu_hat, ms, a_hat, g_hat);
    }
    const double sqrt_gamma_tilde = std::max(std::sqrt(g_hat), 1.0 / std::sqrt(a_hat));
    const double e_nc = std::sqrt(total(S.s[0])), e_r = std::sqrt(total(S.s[2])), e_rs = std::sqrt(total(S.s[5]));
    const double e_df = std::sqrt(total(S.s[3])), e_dfs = std::sqrt(total(S.s[4]));
    const double e_ros = std::sqrt(total(r_os)), e_rsos = std::sqrt(total(rstar_os));
    double result = 0.0;
    switch (which) {
      case 0: case 6: result = e_nc; break;
      case 1: result = e_r; break;
      case 2: result = e_rs; break;
      case 3: case 9: result = e_df; break;
      case 4: result = std::sqrt(total(S.s[8])); break;                                    // swipdg.hh:681-686
      case 5: result = e_nc + e_r + e_df; break;                                           // swipdg.hh:776
      case 7: result = e_ros; break;
      case 8: result = e_rsos; break;
      case 10: result = e_dfs; break;
      case 11: result = (1.0 / std::sqrt(a_bar)) * (std::sqrt(g_bar) * e_nc + e_ros + sqrt_gamma_tilde * e_df); break;      // block-swipdg.hh:791-796
      case 12: result = (1.0 / std::sqrt(a_bar)) * (std::sqrt(g_bar) * e_nc + e_rsos + (1.0 / std::sqrt(a_hat)) * e_dfs); break;  // :962-969
    }
    if (eta) *eta = result;
    if (local_host) {
      if (which == 4 || which == 5) {
        const size_t n = size_t(m->n_own);
        std::vector<double> rows(size_t(9) * n);
        HDD_CUDA(cudaMemcpyAsync(rows.data(), h->ind_out.p, rows.size() * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
        HDD_CUDA(cudaStreamSynchronize(m->stream));
        if (which == 4) {
          const double tot = total(S.s[8]);
          for (size_t k = 0; k < n; ++k) local_host[k] = rows[8 * n + k] / tot;                          // swipdg.hh:709-716
        } else {
          const double tot = std::pow(e_nc + e_r + e_df, 2);
          for (size_t k = 0; k < n; ++k) local_host[k] = 3.0 * (rows[k] + rows[2 * n + k] + rows[3 * n + k]) / tot;  // :807-812
        }
      } else if (which == 11) {
        const double tot = std::pow(result, 2);
        for (int sdm = 0; sdm < ns; ++sdm)                                                                // block-swipdg.hh:870-886
          local_host[sdm] = 3.0 / std::sqrt(a_bar) *
                            (std::sqrt(g_bar) * S.s[0][size_t(sdm)] + r_os[size_t(sdm)] + sqrt_gamma_tilde * S.s[3][size_t(sdm)]) / tot;
      } else if (which == 12) {
        for (int sdm = 0; sdm < ns; ++sdm)                                                                // block-swipdg.hh:1060-1063
          local_host[sdm] = std::sqrt(3.0 / std::sqrt(a_bar) *
                                      (std::sqrt(g_bar) * S.s[0][size_t(sdm)] + rstar_os[size_t(sdm)] + std::sqrt(a_hat) * S.s[4][size_t(sdm)]));
      } else {
        HDD_THROW(HDD_ERR_USING_THIS_WRONG, "Requested type '" << type << "' is not one of available_local()!");
      }
    }
  });
}

}  // extern "C"

// ---- measurement ---------------------------------------------------------------------------------------------------
extern "C" {

int hdd_kernel_bytes(hdd_swipdg* h, int which, double* bytes) {
  return guarded([&] {
    require_init(h);
    const hdd_mesh* m = h->mesh;
    const double cells = double(m->n_own), rows = double(h->n_rows), nnz = double(h->nnz);
    const double geo = m->kind == HDD_SIMPLEX2D ? 48.0 : 32.0, rec = 4.0 * m->nf + 8.0;  // neighbour record + block offset
    const int nl = h->nl;
    double b = 0.0;
    switch (which) {
      case 0: b = 8.0 * nnz + rec * cells + 8.0 * rows /* read p */ + 8.0 * rows /* write q */; break;
      case 1:  // diagonal: read x,p,q,r,dinv, write x,r; block: read x,p,q,r + n_loc^2 block per cell, write x,r,z
        b = uses_block_inverses(h->last_type) ? 7.0 * 8.0 * rows + 8.0 * nl * rows : 7.0 * 8.0 * rows;
        break;
      case 2:  // diagonal: read r,dinv,p, write p; block: read z,p, write p
        b = uses_block_inverses(h->last_type) ? 3.0 * 8.0 * rows : 4.0 * 8.0 * rows;
        break;
      case 3:  // the tensor-grid Q1 kernel reads the neighbour record, the block offset and vertex 0 (28 B), no geometry
        b = 8.0 * nnz + ((m->kind == HDD_CUBE2D && h->polorder == 1 && m->sx > 0) ? 28.0 : geo + rec) * cells;
        break;
      case 4:  // whole estimator pass: Oswald (u 8 B/DoF + incidence 4 B/DoF + 8 B/vertex written and read back) + case 5
      case 5: {  // k_indicators, compulsory traffic: own u, geometry, neighbour ids, vertex ids, 9 rows written
        const double verts = double(m->n_verts_loc);
        const double ind = (8.0 * nl + geo + 4.0 * m->nf + 4.0 * nl + 72.0) * cells + 8.0 * verts;
        const double osw = (8.0 * nl + 4.0 * nl) * cells + (8.0 + 8.0 + 1.0) * verts;
        b = which == 5 ? ind : ind + osw + 72.0 * cells /* rows read by the segmented reduction */;
        break;
      }
      default: HDD_THROW(HDD_ERR_WRONG_INPUT, "unknown kernel id " << which);
    }
    if (bytes) *bytes = b;
  });
}

int hdd_profile_kernel(hdd_swipdg* h, int which, int reps, double* avg_seconds) {
  return guarded([&] {
    require_init(h);
    if (reps < 1) HDD_THROW(HDD_ERR_WRONG_INPUT, "reps must be positive");
    hdd_mesh* m = h->mesh;
    m->set_device();
    cudaStream_t s = m->stream;
    if (which >= 4) {
      check_estimator_space(h);
      if (!h->estimator_vector_resident)
        HDD_THROW(HDD_ERR_USING_THIS_WRONG, "call hdd_estimate once before profiling the estimator kernels");
    } else if (which != 3 && !h->x.p) {
      HDD_THROW(HDD_ERR_USING_THIS_WRONG, "call hdd_solve once before profiling the CG kernels");
    }
    const MeshView v = h->view();
    CgBuffers c{};
    c.values = h->lhs_comps.empty() ? h->lhs_affine->values.p : h->frozen.p;
    c.dinv = h->dinv.p; c.b = h->b.p; c.x = h->x.p; c.r = h->r.p; c.p = h->p.p; c.q = h->q.p;
    c.partial = h->partial.p; c.sc = h->sc.p;
    if (uses_block_inverses(h->last_type)) { c.dinv_block = h->dinv_block.p; c.z = h->z.p; }
    if (which < 3) {
      // un-latch the convergence flag of parity 0 so that the kernels do their work; the vectors are scratch now
      CgScalars sc = *h->sc_host;
      sc.done[0] = 0; sc.done[1] = 0; sc.rz[0] = 1.0; sc.red[0] = 1.0; sc.red[1] = 1.0; sc.max_it = 1 << 30;
      HDD_CUDA(h2d_async(h->sc.p, &sc, sizeof(sc), s));
      h->have_solution = false;
    }
    auto launch = [&]() {
      switch (which) {
        case 0: launch_cg_spmv(v, c, 0, s); break;
        case 1: launch_cg_update(v, c, 0, s); break;
        case 2: launch_cg_direction(v, c, 0, s); break;
        case 3: {
          MatrixPart& part = h->lhs_affine ? *h->lhs_affine : h->lhs_comps[0];
          launch_assemble_lhs(v, h->fn_h(part.factor), part.factor.kind, part.factor.order, h->polorder, part.values.p, s);
          break;
        }
        case 4: indicators_device(h, h->profile_prm, false, 7); break;  // the vector of the last hdd_estimate
        case 5: indicators_device(h, h->profile_prm, false, 2); break;  // k_indicators alone
        default: HDD_THROW(HDD_ERR_WRONG_INPUT, "unknown kernel id " << which);
      }
      if (which == 2) {  // the direction kernel flips the parity state; keep parity 0 alive
        CgScalars sc = *h->sc_host;
        (void)sc;
      }
    };
    for (int k = 0; k < 3; ++k) launch();
    cudaEvent_t e0, e1;
    HDD_CUDA(cudaEventCreate(&e0));
    HDD_CUDA(cudaEventCreate(&e1));
    HDD_CUDA(cudaEventRecord(e0, s));
    for (int k = 0; k < reps; ++k) launch();
    HDD_CUDA(cudaEventRecord(e1, s));
    HDD_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    HDD_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (avg_seconds) *avg_seconds = double(ms) * 1e-3 / reps;
  });
}

int hdd_expression_evaluate(const char* expression, const char* variable, const double* values, int n, double* out) {
  return guarded([&] {
    if (!expression || !variable || !out) HDD_THROW(HDD_ERR_WRONG_INPUT, "NULL argument");
    const Program p = compile_expression(expression, variable);
    double v[4] = {0, 0, 0, 0};
    for (int k = 0; k < n && k < 4; ++k) v[k] = values[k];
    *out = eval_program(p, v);
  });
}

}  // extern "C"
