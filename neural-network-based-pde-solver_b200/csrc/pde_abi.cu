// pde_abi.cu — the extern "C" boundary of libpde_b200.so (see include/pde_b200.h).
// Validates descriptors, plans tile sizes / grids, and enqueues the kernels on the caller's
// stream.  No allocation, no host synchronisation, no global mutable state besides a cached
// copy of the device properties.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <atomic>

#include "../../include/pde_b200.h"
#include "pde_launch.h"
#include "pde_tc.h"

namespace pde {
static std::atomic<unsigned long long> g_launches{0};
static thread_local int g_last_path = -1;
void count_launch(int k) { g_launches.fetch_add((unsigned long long)k, std::memory_order_relaxed); }
void set_last_path(int path) { g_last_path = path; }

DevInfo device_info() {
  // Per-device cache (devices of one box are identical, but be exact).  Threads that fill the same entry at once
  // store the same values; `have` is published last, so a thread that sees it set also sees the attributes.
  static std::atomic<int> sms[64], smem_optin[64], cc_major[64];
  static std::atomic<bool> have[64];
  int dev = 0;
  DevInfo d{0, 0, 0, 0};
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return d; }
  if (!have[dev].load(std::memory_order_acquire)) {
    if (cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return d;
    if (cudaDeviceGetAttribute(&d.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return d;
    if (cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return d;
    sms[dev].store(d.sms, std::memory_order_relaxed);
    smem_optin[dev].store(d.smem_optin, std::memory_order_relaxed);
    cc_major[dev].store(d.cc_major, std::memory_order_relaxed);
    have[dev].store(true, std::memory_order_release);
  }
  return DevInfo{1, sms[dev].load(std::memory_order_relaxed), smem_optin[dev].load(std::memory_order_relaxed),
                 cc_major[dev].load(std::memory_order_relaxed)};
}
}  // namespace pde

namespace {

using namespace pde;

struct Plan {
  int D, order, C, n_lin, n_h, H, Hp, UG, P, KC, pitchP, nthreads, grid, num_tiles, max_grid;
  size_t elem, smem_bytes;
  long long packed_elems, off_W0t, off_b, off_Wt, off_Wn, off_wL, off_bL;
  GradLayout g;
  size_t ws_packed, ws_partial, ws_psums, ws_total;
};

int validate_net(const pde_net* net) {
  if (!net) return PDE_ERR_INVALID;
  if (net->dtype != PDE_F32 && net->dtype != PDE_F64) return PDE_ERR_INVALID;
  if (net->dim < 1 || net->dim > PDE_MAX_DIM) return PDE_ERR_UNSUPPORTED;
  if (net->n_linear < 2 || net->n_linear > PDE_MAX_LINEAR) return PDE_ERR_UNSUPPORTED;
  if (net->activation != PDE_ACT_SIN && net->activation != PDE_ACT_TANH) return PDE_ERR_INVALID;
  if (net->widths[0] != net->dim || net->widths[net->n_linear] != 1) return PDE_ERR_UNSUPPORTED;
  const int H = net->widths[1];
  if (H < 1 || H > PDE_MAX_WIDTH) return PDE_ERR_UNSUPPORTED;
  for (int l = 1; l < net->n_linear; ++l)
    if (net->widths[l] != H) return PDE_ERR_UNSUPPORTED;
  return PDE_OK;
}

// Tile-size / grid planning.  Deterministic in (net geometry, order, n, device), so that
// pde_workspace_bytes and the launches agree.
template <typename T>
int make_plan(const pde_net* net, int order, long long n, Plan* pl) {
  int st = validate_net(net);
  if (st) return st;
  if (order < 0 || order > 2 || n < 1) return PDE_ERR_INVALID;
  DevInfo dv = device_info();
  if (!dv.ok) return PDE_ERR_NO_DEVICE;
  Plan& p = *pl;
  memset(&p, 0, sizeof(p));
  p.elem = sizeof(T);
  p.D = net->dim; p.order = order; p.C = 1 + order * p.D;
  p.n_lin = net->n_linear; p.n_h = p.n_lin - 1; p.H = net->widths[1];
  p.Hp = (int)rup(p.H, 4); if (p.Hp < 8) p.Hp = 8;
  p.UG = p.Hp / 4;
  p.pitchP = p.C * p.Hp + 4;
  {
    long long kc = (32768 / ((long long)p.Hp * (long long)sizeof(T))) & ~3LL;
    if (kc < 4) kc = 4;
    if (kc > p.Hp) kc = p.Hp;
    p.KC = (int)kc;
  }
  // packed parameter layout
  const long long HH = (long long)p.Hp * p.Hp;
  p.off_W0t = 0;
  p.off_b = p.off_W0t + (long long)p.D * p.Hp;
  p.off_Wt = p.off_b + (long long)p.n_h * p.Hp;
  p.off_Wn = p.off_Wt + (long long)(p.n_h - 1) * HH;
  p.off_wL = p.off_Wn + (long long)(p.n_h - 1) * HH;
  p.off_bL = p.off_wL + p.Hp;
  p.packed_elems = rup(p.off_bL + 1, 4);
  p.g = grad_layout(p.D, p.n_h, p.H, p.Hp);

  KernelInfo ki = net_kernel_info<T>(p.D, order);
  if (!ki.fn) return PDE_ERR_UNSUPPORTED;
  int regs = ki.regs > 0 ? ki.regs : 255;
  // registers are allocated per warp in units of 8 per thread
  int regs_alloc = (regs + 7) & ~7;
  int max_threads_regs = (65536 / regs_alloc) & ~31;
  if (max_threads_regs > 1024) max_threads_regs = 1024;

  const int budget1 = dv.smem_optin;                              // one CTA per SM
  const int budget2 = (dv.smem_optin + 1024) / 2 - 1024;          // two CTAs per SM
  auto smem_for = [&](int P) {
    return (size_t)smem_elems<T>(p.D, p.C, p.n_h, p.Hp, p.UG, P, p.KC, p.pitchP) * sizeof(T);
  };
  auto largest_P = [&](int budget, int thread_cap) {
    int best = 0;
    for (int P = 1; P <= 64; ++P) {
      if (P * p.UG > thread_cap) break;
      if ((long long)smem_for(P) > budget) break;
      best = P;
    }
    return best;
  };
  int P1 = largest_P(budget1, max_threads_regs);
  // Wide, deep fp64 nets (d = 5, order 2, 7 hidden layers of 256) leave no room for one point next to the default
  // K-chunk of W: stream W through smaller chunks (multiples of 4) before refusing the shape.
  while (P1 < 1 && p.KC > 4) {
    p.KC -= 4;
    P1 = largest_P(budget1, max_threads_regs);
  }
  if (P1 < 1) return PDE_ERR_UNSUPPORTED;
  int P2 = largest_P(budget2, max_threads_regs / 2 >= p.UG ? max_threads_regs / 2 : p.UG);
  int P = (P2 >= 8) ? P2 : P1;
  // do not make tiles larger than what fills the machine
  long long fill = (n + dv.sms - 1) / dv.sms;
  if (fill < 1) fill = 1;
  if (P > fill) P = (int)fill;
  if (P > 1 && (P & 1) && p.UG < 32) P -= 1;  // keep whole points per warp when UG = 16
  p.P = P;
  p.nthreads = P * p.UG;
  p.smem_bytes = smem_for(P);
  p.num_tiles = (int)((n + P - 1) / P);
  int occ = 1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ki.fn, p.nthreads, p.smem_bytes) != cudaSuccess) {
    cudaGetLastError();
    occ = 1;
  }
  if (occ < 1) occ = 1;
  const size_t pbytes = (size_t)p.g.PP * sizeof(T);
  int cap = pbytes <= (128u << 10) ? 4 : (pbytes <= (512u << 10) ? 2 : 1);
  if (occ > cap) occ = cap;
  p.max_grid = dv.sms * cap;
  long long g = (long long)dv.sms * occ;
  if (g > p.num_tiles) g = p.num_tiles;
  p.grid = (int)g;
  p.ws_packed = (size_t)rup(p.packed_elems * (long long)sizeof(T), 256);
  p.ws_partial = (size_t)rup((long long)p.max_grid * p.g.PP * (long long)sizeof(T), 256);
  p.ws_psums = (size_t)rup((long long)p.max_grid * 8 * (long long)sizeof(double), 256);
  p.ws_total = p.ws_packed + p.ws_partial + p.ws_psums;
  return PDE_OK;
}

int validate_env(const pde_envelope* env) {
  if (!env) return PDE_OK;
  if (env->kind < PDE_ENV_NONE || env->kind > PDE_ENV_EXPWIN) return PDE_ERR_INVALID;
  for (int i = 0; i < PDE_MAX_DIM; ++i)
    if (env->n_nodes[i] < 0 || env->n_nodes[i] > PDE_MAX_NODES) return PDE_ERR_INVALID;
  return PDE_OK;
}

template <typename T>
int run_net(const pde_net* net, int order, int mode, const pde_envelope* env, const pde_program* prog,
            const void* X, long long n, const void* seed, double inv_n, void* J, const void* Jbar, void* sums,
            void* grad, void* energy_grad, void* ws, size_t ws_bytes, cudaStream_t st, const ExchangeReq* ex = nullptr) {
  Plan p;
  int rc = make_plan<T>(net, order, n, &p);
  if (rc) return rc;
  if ((rc = check_ptrs(net))) return rc;
  if (!X || !ws) return PDE_ERR_INVALID;
  if (ws_bytes < p.ws_total) return PDE_ERR_WORKSPACE;
  if ((reinterpret_cast<uintptr_t>(ws) & 15) != 0) return PDE_ERR_INVALID;
  unsigned char* wsb = static_cast<unsigned char*>(ws);
  T* packed = reinterpret_cast<T*>(wsb);
  T* partial = reinterpret_cast<T*>(wsb + p.ws_packed);
  double* psums = reinterpret_cast<double*>(wsb + p.ws_packed + p.ws_partial);
  const bool program = mode == MODE_PROGRAM;
  const int n_q = program ? pde_program_quantities(prog->kind) : 0;
  ReduceArgs<T> r;
  if (mode != MODE_JETS_FWD &&
      (rc = make_reduce_args<T>(p.g, partial, psums, p.grid, 0, n_q, false, static_cast<T*>(grad),
                                program ? static_cast<T*>(sums) : nullptr, program ? static_cast<T*>(energy_grad) : nullptr,
                                ex, &r)))
    return rc;

  PackArgs<T> pa;
  memset(&pa, 0, sizeof(pa));
  for (int l = 0; l < p.n_lin; ++l) { pa.W[l] = static_cast<const T*>(net->W[l]); pa.b[l] = static_cast<const T*>(net->b[l]); }
  pa.n_lin = p.n_lin; pa.D = p.D; pa.H = p.H; pa.Hp = p.Hp; pa.packed = packed;
  pa.off_W0t = p.off_W0t; pa.off_b = p.off_b; pa.off_Wt = p.off_Wt; pa.off_Wn = p.off_Wn;
  pa.off_wL = p.off_wL; pa.off_bL = p.off_bL; pa.total = p.packed_elems;
  if (launch_pack<T>(st, pa) != cudaSuccess) return PDE_ERR_CUDA;

  KArgs<T> a;
  memset(&a, 0, sizeof(a));
  a.n_h = p.n_h; a.H = p.H; a.Hp = p.Hp; a.UG = p.UG; a.act = net->activation;
  a.P = p.P; a.KC = p.KC; a.pitchP = p.pitchP;
  a.packed = packed;
  a.off_W0t = p.off_W0t; a.off_b = p.off_b; a.off_Wt = p.off_Wt; a.off_Wn = p.off_Wn; a.off_wL = p.off_wL; a.off_bL = p.off_bL;
  a.X = static_cast<const T*>(X); a.n = n; a.num_tiles = p.num_tiles;
  a.mode = mode; a.want_grad = (grad != nullptr) || (energy_grad != nullptr);
  a.J = static_cast<T*>(J); a.Jbar = static_cast<const T*>(Jbar);
  a.n_q = n_q;
  if (program) {
    a.prog = prog->kind;
    fill_env<T>(env, &a.env);
    a.alpha = (T)prog->alpha; a.beta_const = (T)prog->beta_const; a.energy_const = (T)prog->energy_const;
    a.inv_n = (T)inv_n;
    a.f = static_cast<const T*>(prog->f); a.beta = static_cast<const T*>(prog->beta);
    a.energy = static_cast<const T*>(prog->energy); a.seed = static_cast<const T*>(seed);
    a.faces = prog->faces; a.face_n = flux_face_n(prog, n);
  }
  a.partial = partial; a.psums = psums; a.PP = p.g.PP;
  a.off_gW0 = p.g.off_gW0; a.off_gb0 = p.g.off_gb0; a.off_gW = p.g.off_gW; a.off_gwL = p.g.off_gwL; a.off_gbL = p.g.off_gbL;
  if (launch_net<T>(p.D, order, p.grid, p.nthreads, p.smem_bytes, st, a) != cudaSuccess) return PDE_ERR_CUDA;
  set_last_path(0);

  if (mode == MODE_JETS_FWD) return PDE_OK;
  if (launch_reduce<T>(st, r) != cudaSuccess) return PDE_ERR_CUDA;
  return PDE_OK;
}

template <typename T>
cudaError_t run_wan(const pde_wan* wan, const void* X, long long n, const void* Ju, const void* Jv, const void* seed,
                    double inv_n, void* sums, void* Jbar_u, void* Jbar_v, void* workspace, int blocks, cudaStream_t st) {
  WanArgs<T> a;
  memset(&a, 0, sizeof(a));
  a.D = wan->dim; a.n = n;
  a.X = static_cast<const T*>(X); a.Ju = static_cast<const T*>(Ju); a.Jv = static_cast<const T*>(Jv);
  a.f = static_cast<const T*>(wan->f); a.beta = static_cast<const T*>(wan->beta);
  a.energy = static_cast<const T*>(wan->energy); a.seed = static_cast<const T*>(seed);
  a.alpha = (T)wan->alpha; a.beta_const = (T)wan->beta_const; a.energy_const = (T)wan->energy_const;
  a.w_lo = (T)wan->w_lo; a.w_hi = (T)wan->w_hi; a.eps_den = (T)wan->eps_den; a.inv_n = (T)inv_n;
  fill_env<T>(&wan->env_u, &a.env_u); fill_env<T>(&wan->env_v, &a.env_v);
  a.Jbar_u = static_cast<T*>(Jbar_u); a.Jbar_v = static_cast<T*>(Jbar_v);
  a.psums = static_cast<double*>(workspace); a.sums = static_cast<T*>(sums); a.blocks = blocks;
  return launch_wan<T>(st, a);
}

}  // namespace

extern "C" {

int pde_abi_version(void) { return PDE_ABI_VERSION; }

const char* pde_strerror(int status) {
  switch (status) {
    case PDE_OK: return "ok";
    case PDE_ERR_INVALID: return "invalid argument";
    case PDE_ERR_UNSUPPORTED: return "unsupported network / program shape";
    case PDE_ERR_WORKSPACE: return "workspace too small";
    case PDE_ERR_CUDA: return "CUDA runtime error";
    case PDE_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
    default: return "unknown status";
  }
}

int pde_param_count(const pde_net* net, int64_t* n_params) {
  int st = validate_net(net);
  if (st) return st;
  if (!n_params) return PDE_ERR_INVALID;
  *n_params = param_count(net->dim, net->n_linear - 1, net->widths[1]);
  return PDE_OK;
}

int pde_jet_channels(int32_t dim, int32_t order) {
  if (dim < 1 || dim > PDE_MAX_DIM || order < 0 || order > 2) return PDE_ERR_INVALID;
  return 1 + order * dim;
}

int pde_program_quantities(int32_t kind) {
  switch (kind) {
    case PDE_PROG_PINN: case PDE_PROG_DRM: case PDE_PROG_MSE: case PDE_PROG_FLUX: return 1;
    case PDE_PROG_RAYLEIGH: return 2;
    default: return PDE_ERR_INVALID;
  }
}

int pde_program_order(int32_t kind) {
  switch (kind) {
    case PDE_PROG_PINN: return 2;
    case PDE_PROG_DRM: case PDE_PROG_RAYLEIGH: case PDE_PROG_FLUX: return 1;
    case PDE_PROG_MSE: return 0;
    default: return PDE_ERR_INVALID;
  }
}

int pde_workspace_bytes(const pde_net* net, int32_t order, int64_t n_points, size_t* bytes) {
  if (!bytes) return PDE_ERR_INVALID;
  Plan p;
  int rc = (net && net->dtype == PDE_F64) ? make_plan<double>(net, order, n_points, &p)
                                          : make_plan<float>(net, order, n_points, &p);
  if (rc) return rc;
  size_t need = p.ws_total;
  size_t tc = 0;
  if (pde::tc_workspace_bytes(net, order, n_points, &tc) == PDE_OK && tc > need) need = tc;
  *bytes = need;
  return PDE_OK;
}

int pde_jets_forward(const pde_net* net, int32_t order, const void* X, int64_t n_points, void* J,
                     void* workspace, size_t workspace_bytes, void* stream) {
  if (!net || !J) return PDE_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = pde::tc_jets_forward(net, order, X, n_points, J, workspace, workspace_bytes, st);
  if (rc != PDE_ERR_UNSUPPORTED) return rc;
  if (net->dtype == PDE_F64)
    return run_net<double>(net, order, MODE_JETS_FWD, nullptr, nullptr, X, n_points, nullptr, 1.0, J, nullptr, nullptr,
                           nullptr, nullptr, workspace, workspace_bytes, st);
  return run_net<float>(net, order, MODE_JETS_FWD, nullptr, nullptr, X, n_points, nullptr, 1.0, J, nullptr, nullptr,
                        nullptr, nullptr, workspace, workspace_bytes, st);
}

int pde_jets_backward(const pde_net* net, int32_t order, const void* X, int64_t n_points, const void* Jbar,
                      void* grad, void* workspace, size_t workspace_bytes, void* stream) {
  if (!net || !Jbar || !grad) return PDE_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = pde::tc_jets_backward(net, order, X, n_points, Jbar, grad, workspace, workspace_bytes, st);
  if (rc != PDE_ERR_UNSUPPORTED) return rc;
  if (net->dtype == PDE_F64)
    return run_net<double>(net, order, MODE_JETS_BWD, nullptr, nullptr, X, n_points, nullptr, 1.0, nullptr, Jbar,
                           nullptr, grad, nullptr, workspace, workspace_bytes, st);
  return run_net<float>(net, order, MODE_JETS_BWD, nullptr, nullptr, X, n_points, nullptr, 1.0, nullptr, Jbar, nullptr,
                        grad, nullptr, workspace, workspace_bytes, st);
}

static int residual_loss_grad_impl(const pde_net* net, const pde_envelope* env, const pde_program* prog, const void* X,
                                   int64_t n_points, const void* seed, double inv_n, void* sums, void* grad,
                                   void* energy_grad, void* workspace, size_t workspace_bytes, void* stream,
                                   const ExchangeReq* ex) {
  if (!net || !prog) return PDE_ERR_INVALID;
  const int order = pde_program_order(prog->kind);
  if (order < 0) return PDE_ERR_INVALID;
  int rc = validate_env(env);
  if (rc) return rc;
  if (!sums && !grad && !energy_grad) return PDE_ERR_INVALID;
  if (prog->kind == PDE_PROG_FLUX) {   // the face mask and the block layout of the points (include/pde_b200.h)
    if (net->dim < 1 || net->dim > PDE_MAX_DIM) return PDE_ERR_UNSUPPORTED;
    if (prog->faces <= 0 || prog->faces >= (1 << (2 * net->dim))) return PDE_ERR_INVALID;
    if (n_points % __builtin_popcount((unsigned)prog->faces) != 0) return PDE_ERR_INVALID;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Blackwell tensor-core path for the shapes it covers (fp32, H = 64 sin/tanh nets); it
  // declines with PDE_ERR_UNSUPPORTED and the generic SIMT kernel takes over.
  rc = pde::tc_residual_loss_grad(net, env, prog, X, n_points, seed, inv_n, sums, grad, energy_grad, workspace,
                                  workspace_bytes, st, ex);
  if (rc != PDE_ERR_UNSUPPORTED) return rc;
  if (net->dtype == PDE_F64)
    return run_net<double>(net, order, MODE_PROGRAM, env, prog, X, n_points, seed, inv_n, nullptr, nullptr, sums, grad,
                           energy_grad, workspace, workspace_bytes, st, ex);
  return run_net<float>(net, order, MODE_PROGRAM, env, prog, X, n_points, seed, inv_n, nullptr, nullptr, sums, grad,
                        energy_grad, workspace, workspace_bytes, st, ex);
}

int pde_residual_loss_grad(const pde_net* net, const pde_envelope* env, const pde_program* prog, const void* X,
                           int64_t n_points, const void* seed, double inv_n, void* sums, void* grad,
                           void* energy_grad, void* workspace, size_t workspace_bytes, void* stream) {
  return residual_loss_grad_impl(net, env, prog, X, n_points, seed, inv_n, sums, grad, energy_grad, workspace,
                                 workspace_bytes, stream, nullptr);
}

int pde_residual_loss_grad_exchange(const pde_net* net, const pde_envelope* env, const pde_program* prog, const void* X,
                                    int64_t n_points, const void* seed, double inv_n, void* result, void* workspace,
                                    size_t workspace_bytes, const pde_peers* peers, int64_t slot_elems, void* seq,
                                    void* stream) {
  if (!net || !prog || !result || !peers || !seq) return PDE_ERR_INVALID;
  int64_t np = 0;
  int rc = pde_param_count(net, &np);
  if (rc) return rc;
  const int K = pde_program_quantities(prog->kind);
  if (K < 1) return PDE_ERR_INVALID;
  const size_t es = net->dtype == PDE_F64 ? 8 : 4;
  unsigned char* base = static_cast<unsigned char*>(result);
  ExchangeReq ex{peers, slot_elems, seq};
  return residual_loss_grad_impl(net, env, prog, X, n_points, seed, inv_n, base + (size_t)(np + 1) * es, base,
                                 base + (size_t)np * es, workspace, workspace_bytes, stream, &ex);
}

int pde_query_path(const pde_net* net, const pde_program* prog, int64_t n_points) {
  int st = validate_net(net);
  if (st) return st;
  if (!prog) return PDE_ERR_INVALID;
  return pde::tc_supported(net, prog, n_points) ? 1 : 0;
}

int pde_query_jets_path(const pde_net* net, int32_t order, int64_t n_points) {
  int st = validate_net(net);
  if (st) return st;
  return pde::tc_jets_supported(net, order, n_points) ? 1 : 0;
}

int pde_set_kernel_path(int32_t path) {
  if (path < -1 || path > 1) return PDE_ERR_INVALID;
  pde::tc_set_path_override(path);
  return PDE_OK;
}

int pde_kernel_path(void) { return pde::tc_get_path_override(); }

int pde_last_kernel_path(void) { return pde::g_last_path; }

uint64_t pde_launch_count(void) { return pde::g_launches.load(std::memory_order_relaxed); }

int pde_wan_pointwise(const pde_wan* wan, const void* X, int64_t n_points, const void* Ju, const void* Jv,
                      const void* seed, double inv_n, void* sums, void* Jbar_u, void* Jbar_v, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if (!wan || !X || !Ju || !Jv || !sums || !workspace || n_points < 1) return PDE_ERR_INVALID;
  if (wan->dim < 1 || wan->dim > PDE_MAX_DIM) return PDE_ERR_UNSUPPORTED;
  if (wan->dtype != PDE_F32 && wan->dtype != PDE_F64) return PDE_ERR_INVALID;
  int rc = validate_env(&wan->env_u);
  if (rc) return rc;
  if ((rc = validate_env(&wan->env_v))) return rc;
  DevInfo dv = device_info();
  if (!dv.ok) return PDE_ERR_NO_DEVICE;
  int blocks = (int)((n_points + 255) / 256);
  if (blocks > dv.sms * 4) blocks = dv.sms * 4;
  if (workspace_bytes < (size_t)blocks * 8 * sizeof(double)) return PDE_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const cudaError_t err =
      wan->dtype == PDE_F64
          ? run_wan<double>(wan, X, n_points, Ju, Jv, seed, inv_n, sums, Jbar_u, Jbar_v, workspace, blocks, st)
          : run_wan<float>(wan, X, n_points, Ju, Jv, seed, inv_n, sums, Jbar_u, Jbar_v, workspace, blocks, st);
  return err == cudaSuccess ? PDE_OK : PDE_ERR_CUDA;
}

}  // extern "C"
