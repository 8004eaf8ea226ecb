// pde_launch.h — host-side launch shims between the C ABI (pde_abi.cu) and the per-dtype
// instantiation units (pde_f32.cu / pde_f64.cu), and the planning helpers that the generic
// (pde_abi.cu) and tensor-core (pde_tc.cu) launch sequences share.
#pragma once
#include <cuda_runtime.h>
#include <string.h>
#include "pde_simt.cuh"
#include "pde_tc.h"

namespace pde {

// Process-wide counters the host side reads through the C ABI (pde_launch_count, pde_last_kernel_path): every kernel
// this library enqueues is counted where it is launched, and the fused calls record which kernel family served them.
void count_launch(int k = 1);
void set_last_path(int path);   // 0 generic SIMT kernel, 1 tcgen05 kernel

// Attributes of the current device, cached per device ordinal (safe to call from several host threads); ok = 0 when
// there is no usable device.
struct DevInfo {
  int ok, sms, smem_optin, cc_major;
};
DevInfo device_info();

inline long long rup(long long x, long long m) { return (x + m - 1) / m * m; }

// Scalar parameters of a network [D, H, ..., H, 1] with n_h hidden layers: W0 [H][D], b0 [H], (n_h - 1) x (W [H][H],
// b [H]), wL [H], bL.
inline long long param_count(long long D, long long n_h, long long H) {
  return H * D + H + (n_h - 1) * (H * H + H) + H + 1;
}

inline int check_ptrs(const pde_net* net) {
  for (int l = 0; l < net->n_linear; ++l)
    if (!net->W[l] || !net->b[l]) return PDE_ERR_INVALID;
  return PDE_OK;
}

// Points per face of a PDE_PROG_FLUX batch of n points (0 for every other program).  The mask is validated first.
inline long long flux_face_n(const pde_program* prog, long long n) {
  return prog->kind == PDE_PROG_FLUX ? n / __builtin_popcount((unsigned)prog->faces) : 0;
}

template <typename T>
void fill_env(const pde_envelope* env, EnvDev<T>* e) {
  memset(e, 0, sizeof(*e));
  if (!env) return;
  e->kind = env->kind;
  e->lo = (T)env->lo; e->hi = (T)env->hi;
  for (int i = 0; i < PDE_MAX_DIM; ++i) {
    e->n_nodes[i] = env->n_nodes[i];
    for (int k = 0; k < PDE_MAX_NODES; ++k) e->nodes[i][k] = (T)env->nodes[i][k];
  }
}

// Per-CTA partial-gradient vector: the natural parameter order with the hidden width padded to Hp (W0 [Hp][D], b0,
// (n_h - 1) x (W [Hp][Hp], b), wL, bL), PP elements per CTA.  n_params counts the unpadded parameters.
struct GradLayout {
  int D, n_lin, H, Hp;
  long long off_gW0, off_gb0, off_gW, off_gwL, off_gbL, PP, n_params;
};

inline GradLayout grad_layout(int D, int n_h, int H, int Hp) {
  GradLayout g;
  g.D = D; g.n_lin = n_h + 1; g.H = H; g.Hp = Hp;
  g.off_gW0 = 0;
  g.off_gb0 = (long long)Hp * D;
  g.off_gW = g.off_gb0 + Hp;
  g.off_gwL = g.off_gW + (long long)(n_h - 1) * ((long long)Hp * Hp + Hp);
  g.off_gbL = g.off_gwL + Hp;
  g.PP = rup(g.off_gbL + 1, 4);
  g.n_params = param_count(D, n_h, H);
  return g;
}

// Arguments of reduce_kernel: `grid` partial vectors laid out as `g`, `psum_grid` rows of psums (0: grid rows); each
// output may be null.  With an exchange, every reduced element is summed over the ranks before it is written; what is
// exchanged is the caller's whole [grad | dE | sums] row, so all three outputs must be given.  Returns a status.
template <typename T>
int make_reduce_args(const GradLayout& g, const T* partial, const double* psums, int grid, int psum_grid, int n_q,
                     bool accumulate, T* grad, T* sums, T* energy_grad, const ExchangeReq* ex, ReduceArgs<T>* r) {
  memset(r, 0, sizeof(*r));
  r->partial = partial; r->psums = psums; r->PP = g.PP; r->grid = grid; r->psum_grid = psum_grid;
  r->n_lin = g.n_lin; r->D = g.D; r->H = g.H; r->Hp = g.Hp; r->n_q = n_q;
  r->off_gW0 = g.off_gW0; r->off_gb0 = g.off_gb0; r->off_gW = g.off_gW; r->off_gwL = g.off_gwL; r->off_gbL = g.off_gbL;
  r->n_params = g.n_params;
  r->grad = grad; r->sums = sums; r->energy_grad = energy_grad;
  r->accumulate = accumulate ? 1 : 0;
  if (ex) {
    if (!grad || !sums || !energy_grad) return PDE_ERR_INVALID;
    const int rc = comm_fill_args(ex->peers, sizeof(T) == 8 ? PDE_F64 : PDE_F32, g.n_params + 1 + n_q, ex->slot_elems,
                                  ex->seq, &r->comm);
    if (rc) return rc;
    r->have_comm = 1;
  }
  return PDE_OK;
}

struct KernelInfo {
  const void* fn;
  int regs;
  int max_threads;   // cudaFuncAttributes::maxThreadsPerBlock, the largest block a launch accepts (0: unknown)
};

// kernel handle for (dim, order); nullptr if out of range
template <typename T> KernelInfo net_kernel_info(int dim, int order);
template <typename T> cudaError_t launch_net(int dim, int order, int grid, int block, size_t smem, cudaStream_t st, const KArgs<T>& a);
template <typename T> cudaError_t launch_pack(cudaStream_t st, const PackArgs<T>& a);
template <typename T> cudaError_t launch_reduce(cudaStream_t st, const ReduceArgs<T>& a);

// WAN elementwise coupling on jets (pde_wan in include/pde_b200.h)
template <typename T>
struct WanArgs {
  int D;
  long long n;
  const T* X; const T* Ju; const T* Jv;
  const T* f; const T* beta; const T* energy; const T* seed;
  T alpha, beta_const, energy_const, w_lo, w_hi, eps_den, inv_n;
  EnvDev<T> env_u, env_v;
  T* Jbar_u; T* Jbar_v;
  double* psums;   // [blocks][8]
  T* sums;         // (5) out, written by the finishing kernel
  int blocks;
};
template <typename T> cudaError_t launch_wan(cudaStream_t st, const WanArgs<T>& a);

}  // namespace pde
