// pde_step.cu — the device-side pieces of a training epoch that sit around the loss step
// (SURVEY.md §8f-1, §8f-3): collocation-point sampling with the manufactured right-hand side,
// fused Adam over the flat gradient vector the loss step writes, and device-side best-model
// tracking.  All of them are single launches on the caller's stream without host synchronisation,
// so an epoch (sample -> loss step -> Adam -> evaluation -> keep-best) is one CUDA graph.
//
// Reference behaviour restated here:
//   sample_interior            Poisson_ND.py:187-190   X = rand(N, d) * L
//   exact_u_prod_sin / rhs_f   Poisson_ND.py:49-58     u* = prod_i sin(k_i pi x_i / L),  f = sum_i (k_i pi / L)^2 u*
//   torch.optim.Adam(lr)       Poisson_ND.py:177,240   default betas (0.9, 0.999), eps 1e-8, no weight decay
//   best-model tracking        Poisson_ND.py:288-300   if l2 < best_l2: keep a copy of the parameters
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/pde_b200.h"
#include "pde_launch.h"

namespace {

// ---------------------------------------------------------------- Philox4x32-10 (counter-based, stateless)
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0; key.y += W1;
  }
  return ctr;
}

template <typename T> __device__ __forceinline__ T sin_(T x);
template <> __device__ __forceinline__ float sin_<float>(float x) { return sinf(x); }
template <> __device__ __forceinline__ double sin_<double>(double x) { return sin(x); }
template <typename T> __device__ __forceinline__ T cos_(T x);
template <> __device__ __forceinline__ float cos_<float>(float x) { return cosf(x); }
template <> __device__ __forceinline__ double cos_<double>(double x) { return cos(x); }

template <typename T> __device__ __forceinline__ T below_(T hi, T lo);
template <> __device__ __forceinline__ float below_<float>(float hi, float lo) { return nextafterf(hi, lo); }
template <> __device__ __forceinline__ double below_<double>(double hi, double lo) { return nextafter(hi, lo); }

// uniform in [0, 1): 24 random bits for float, 53 for double (the resolution torch.rand uses)
__device__ __forceinline__ float unit_f32(uint32_t a) { return (float)(a >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ double unit_f64(uint32_t a, uint32_t b) {
  const unsigned long long v = ((unsigned long long)(a >> 6) << 27) | (unsigned long long)(b >> 5);   // 26 + 27 bits
  return (double)v * (1.0 / 9007199254740992.0);
}

struct SampleArgs {
  int dim;
  long long n;
  double lo, hi, period;
  unsigned long long seed, offset;
  int have_k;
  double k[PDE_MAX_DIM];
  void* X; void* u; void* f;
  const void* X_in;   // evaluate the manufactured solution at given points instead of sampling
  const long long* offset_add;   // device, optional: added to `offset` (e.g. the optimiser's step counter)
  int faces;          // sample_faces_kernel: face mask, points per face, and the Neumann data out (the u slot is unused)
  long long face_n;
  void* g;
};

// The coordinates of point p: Philox counters (point index | coordinate group << 62, call offset), uniform in
// [lo, hi) with the half-open interval kept through rounding (float: (hi - lo) * (1 - 2^-24) may round to hi - lo).
template <typename T>
__device__ __forceinline__ void draw_point(const SampleArgs& a, long long p, uint2 key, unsigned long long off, T (&x)[PDE_MAX_DIM]) {
  if (sizeof(T) == 4) {
    for (int c = 0; 4 * c < a.dim; ++c) {
      const uint4 r = philox4x32_10(make_uint4((uint32_t)p, (uint32_t)(p >> 32) | ((uint32_t)c << 30), (uint32_t)off, (uint32_t)(off >> 32)), key);
      const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
      for (int e = 0; e < 4 && 4 * c + e < a.dim; ++e) x[4 * c + e] = (T)(a.lo + (a.hi - a.lo) * (double)unit_f32(rr[e]));
    }
  } else {
    for (int c = 0; 2 * c < a.dim; ++c) {
      const uint4 r = philox4x32_10(make_uint4((uint32_t)p, (uint32_t)(p >> 32) | ((uint32_t)c << 30), (uint32_t)off, (uint32_t)(off >> 32)), key);
      x[2 * c] = (T)(a.lo + (a.hi - a.lo) * unit_f64(r.x, r.y));
      if (2 * c + 1 < a.dim) x[2 * c + 1] = (T)(a.lo + (a.hi - a.lo) * unit_f64(r.z, r.w));
    }
  }
  for (int i = 0; i < a.dim; ++i)
    if (x[i] >= (T)a.hi) x[i] = below_<T>((T)a.hi, (T)a.lo);
}

// One thread per point: coordinates from Philox counters (point index | coordinate group << 62, call offset),
// written row-major; u* and f in the same pass.  HBM-bound: 4 (d + 2) bytes per point.
template <typename T>
__global__ void sample_rhs_kernel(const SampleArgs a) {
  T* X = static_cast<T*>(a.X);
  const T* Xin = static_cast<const T*>(a.X_in);
  T* U = static_cast<T*>(a.u);
  T* F = static_cast<T*>(a.f);
  const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
  const unsigned long long off = a.offset + (a.offset_add ? (unsigned long long)*a.offset_add : 0ull);
  T s = T(0);
  if (a.have_k) {
    for (int i = 0; i < a.dim; ++i) {
      const T w = (T)(a.k[i] * 3.14159265358979323846) / (T)a.period;
      s += w * w;
    }
  }
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < a.n; p += (long long)gridDim.x * blockDim.x) {
    T x[PDE_MAX_DIM];
    if (Xin) {
      for (int i = 0; i < a.dim; ++i) x[i] = Xin[p * a.dim + i];
    } else {
      draw_point<T>(a, p, key, off, x);
      for (int i = 0; i < a.dim; ++i) X[p * a.dim + i] = x[i];
    }
    if (a.have_k && (U || F)) {
      T u = T(1);
      for (int i = 0; i < a.dim; ++i) u *= sin_<T>((T)(a.k[i] * 3.14159265358979323846) * x[i] / (T)a.period);
      if (U) U[p] = u;
      if (F) F[p] = s * u;
    }
  }
}

// Face points (include/pde_b200.h, pde_sample_faces_rhs): the coordinates sample_rhs_kernel draws for the same point
// index, the block's face coordinate set to lo or hi, and the outward normal derivative of u* in the same pass.
// HBM-bound: 4 (d + 1) bytes per point.
template <typename T>
__global__ void sample_faces_kernel(const SampleArgs a) {
  T* X = static_cast<T*>(a.X);
  T* G = static_cast<T*>(a.g);
  const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
  const unsigned long long off = a.offset + (a.offset_add ? (unsigned long long)*a.offset_add : 0ull);
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < a.n; p += (long long)gridDim.x * blockDim.x) {
    T x[PDE_MAX_DIM];
    draw_point<T>(a, p, key, off, x);
    int ax, sg;
    pde::flux_face(a.faces, a.face_n, p, ax, sg);
    for (int i = 0; i < a.dim; ++i) {
      if (i == ax) x[i] = (T)(sg > 0 ? a.hi : a.lo);
      X[p * a.dim + i] = x[i];
    }
    if (G) {
      T v = T(1);
      for (int i = 0; i < a.dim; ++i) {
        const T w = (T)(a.k[i] * 3.14159265358979323846) / (T)a.period;
        const T z = (T)(a.k[i] * 3.14159265358979323846) * x[i] / (T)a.period;
        v *= (i == ax) ? w * cos_<T>(z) : sin_<T>(z);
      }
      G[p] = sg > 0 ? v : -v;
    }
  }
}

// ---------------------------------------------------------------- fused Adam
struct AdamArgs {
  int n_tensors;
  void* param[2 * PDE_MAX_LINEAR + 1];
  long long start[2 * PDE_MAX_LINEAR + 2];   // prefix sums of numel
  double lr, beta1, beta2, eps, weight_decay, grad_scale;
  const void* grad; void* m; void* v;
  const long long* step;   // device: number of steps taken so far
};

template <typename T>
__global__ void adam_kernel(const AdamArgs a) {
  const long long total = a.start[a.n_tensors];
  const double t = (double)(*a.step + 1);
  // torch.optim.Adam (single-tensor path): step_size = lr / (1 - beta1^t), denom = sqrt(v) / sqrt(1 - beta2^t) + eps
  const double bc1 = 1.0 - pow(a.beta1, t), bc2 = 1.0 - pow(a.beta2, t);
  const T step_size = (T)(a.lr / bc1), rs2 = (T)(1.0 / sqrt(bc2));
  const T b1 = (T)a.beta1, b2 = (T)a.beta2, eps = (T)a.eps, wd = (T)a.weight_decay, gs = (T)a.grad_scale;
  const T* G = static_cast<const T*>(a.grad);
  T* M = static_cast<T*>(a.m);
  T* V = static_cast<T*>(a.v);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int k = 0;
    while (i >= a.start[k + 1]) ++k;
    T* p = static_cast<T*>(a.param[k]) + (i - a.start[k]);
    T g = G[i] * gs;
    const T w = *p;
    if (wd != T(0)) g += wd * w;
    const T m = M[i] + (T(1) - b1) * (g - M[i]);            // lerp, as torch does
    const T v = b2 * V[i] + (T(1) - b2) * g * g;
    M[i] = m; V[i] = v;
    *p = w - step_size * (m / (sqrt(v) * rs2 + eps));
  }
}

__global__ void bump_step_kernel(long long* step) { *step += 1; }

// ---------------------------------------------------------------- keep the best parameters (device-side)
struct BestArgs {
  int n_tensors;
  const void* param[2 * PDE_MAX_LINEAR + 1];
  long long start[2 * PDE_MAX_LINEAR + 2];
  const void* metric; void* best_metric; void* best_flat;
  long long* best_step; const long long* step;
};

template <typename T>
__global__ void keep_best_kernel(const BestArgs a) {
  __shared__ int take;
  if (threadIdx.x == 0) {
    const T m = *static_cast<const T*>(a.metric);
    T* b = static_cast<T*>(a.best_metric);
    take = (m < *b) ? 1 : 0;     // NaN never wins
    if (take) {
      *b = m;
      if (a.best_step && a.step) *a.best_step = *a.step;
    }
  }
  __syncthreads();
  if (!take) return;
  T* out = static_cast<T*>(a.best_flat);
  const long long total = a.start[a.n_tensors];
  for (long long i = threadIdx.x; i < total; i += blockDim.x) {
    int k = 0;
    while (i >= a.start[k + 1]) ++k;
    out[i] = static_cast<const T*>(a.param[k])[i - a.start[k]];
  }
}

int grid_for(long long n, int block) {
  long long g = (n + block - 1) / block;
  return (int)(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));
}

// The scalar end of the WAN losses: (loss_pde, loss_v, loss_norm, total) of the four means and the 4 x 4 Jacobian
// d out_i / d mean_j, one thread.  The reference evaluates these with ~25 separate 0-d tensor operations per call
// (Poisson_ND.py:118-127, IPW_1D_WAN.py:108-114, QHO_2D.py:218-224, KH_1D.py:263-268), which at 1000 points costs as
// much as the network sweeps.
struct WanScalarArgs {
  int kind;
  double eps_pde, eps_log, vol, reg, w_pde, w_norm;
  const void* m;
  void* out;
  void* jac;
};
template <typename T>
__global__ void wan_scalars_kernel(const WanScalarArgs a) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const T* m = static_cast<const T*>(a.m);
  T* out = static_cast<T*>(a.out);
  T* J = static_cast<T*>(a.jac);
  const T m0 = m[0], m1 = m[1], m2 = m[2], m3 = m[3];
  const T e1 = (T)a.eps_pde, e2 = (T)a.eps_log, vol = (T)a.vol, reg = (T)a.reg, wp = (T)a.w_pde, wn = (T)a.w_norm;
  T pde, d0, d1;
  if (a.kind == 0) {          // weak^2 / (norm_phi + eps)
    const T den = m1 + e1;
    pde = m0 * m0 / den;
    d0 = T(2) * m0 / den;
    d1 = -(m0 * m0) / (den * den);
  } else {                    // KH: (vol * weak / (vol * norm_phi + eps))^2
    const T I = vol * m0, den = vol * m1 + e1, r = I / den;
    pde = r * r;
    d0 = T(2) * r * vol / den;
    d1 = -T(2) * r * I * vol / (den * den);
  }
  const T k = -T(1) / (pde + e2);
  const T lv = -log(pde + e2) + reg * m3;
  const T nv = vol * m2 - T(1);
  for (int i = 0; i < 16; ++i) J[i] = T(0);
  out[0] = pde;             J[0] = d0;          J[1] = d1;
  out[1] = lv;              J[4] = k * d0;      J[5] = k * d1;      J[7] = reg;
  out[2] = nv * nv;         J[10] = T(2) * nv * vol;
  out[3] = wp * pde + wn * nv * nv;
  J[12] = wp * d0;          J[13] = wp * d1;    J[14] = wn * T(2) * nv * vol;
}

}  // namespace

extern "C" {

int pde_wan_scalars(int32_t dtype, int32_t kind, const void* means, const double* consts, void* out, void* jac, void* stream) {
  if ((dtype != PDE_F32 && dtype != PDE_F64) || kind < 0 || kind > 1 || !means || !consts || !out || !jac) return PDE_ERR_INVALID;
  WanScalarArgs a;
  a.kind = kind;
  a.eps_pde = consts[0]; a.eps_log = consts[1]; a.vol = consts[2]; a.reg = consts[3]; a.w_pde = consts[4]; a.w_norm = consts[5];
  a.m = means; a.out = out; a.jac = jac;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == PDE_F32) wan_scalars_kernel<float><<<1, 32, 0, st>>>(a);
  else wan_scalars_kernel<double><<<1, 32, 0, st>>>(a);
  pde::count_launch(1);
  return cudaGetLastError() == cudaSuccess ? PDE_OK : PDE_ERR_CUDA;
}

int pde_sample_points_rhs(int32_t dtype, int32_t dim, int64_t n_points, double lo, double hi, uint64_t seed,
                          uint64_t offset, const void* offset_add, const double* k, double period, const void* X_in,
                          void* X, void* u_exact, void* f, void* stream) {
  if (dtype != PDE_F32 && dtype != PDE_F64) return PDE_ERR_INVALID;
  if (dim < 1 || dim > PDE_MAX_DIM) return PDE_ERR_UNSUPPORTED;
  if (n_points < 1 || !(hi > lo)) return PDE_ERR_INVALID;
  if (!X_in && !X) return PDE_ERR_INVALID;
  if ((u_exact || f) && (!k || !(period > 0.0))) return PDE_ERR_INVALID;
  SampleArgs a;
  a.dim = dim; a.n = n_points; a.lo = lo; a.hi = hi; a.period = period > 0.0 ? period : 1.0;
  a.seed = seed; a.offset = offset; a.have_k = k ? 1 : 0;
  for (int i = 0; i < PDE_MAX_DIM; ++i) a.k[i] = (k && i < dim) ? k[i] : 0.0;
  a.X = X; a.u = u_exact; a.f = f; a.X_in = X_in; a.offset_add = static_cast<const long long*>(offset_add);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int block = 256, grid = grid_for(n_points, block);
  if (dtype == PDE_F32) sample_rhs_kernel<float><<<grid, block, 0, st>>>(a);
  else sample_rhs_kernel<double><<<grid, block, 0, st>>>(a);
  pde::count_launch(1);
  return cudaGetLastError() == cudaSuccess ? PDE_OK : PDE_ERR_CUDA;
}

int pde_sample_faces_rhs(int32_t dtype, int32_t dim, int64_t n_per_face, int32_t faces, double lo, double hi,
                         uint64_t seed, uint64_t offset, const void* offset_add, const double* k, double period, void* X,
                         void* g, void* stream) {
  if (dtype != PDE_F32 && dtype != PDE_F64) return PDE_ERR_INVALID;
  if (dim < 1 || dim > PDE_MAX_DIM) return PDE_ERR_UNSUPPORTED;
  if (faces <= 0 || faces >= (1 << (2 * dim)) || n_per_face < 1 || !(hi > lo) || !X) return PDE_ERR_INVALID;
  if (g && (!k || !(period > 0.0))) return PDE_ERR_INVALID;
  SampleArgs a;
  memset(&a, 0, sizeof(a));
  a.dim = dim; a.n = n_per_face * __builtin_popcount((unsigned)faces); a.lo = lo; a.hi = hi;
  a.period = period > 0.0 ? period : 1.0;
  a.seed = seed; a.offset = offset; a.have_k = k ? 1 : 0;
  for (int i = 0; i < PDE_MAX_DIM; ++i) a.k[i] = (k && i < dim) ? k[i] : 0.0;
  a.X = X; a.g = g; a.offset_add = static_cast<const long long*>(offset_add);
  a.faces = faces; a.face_n = n_per_face;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int block = 256, grid = grid_for(a.n, block);
  if (dtype == PDE_F32) sample_faces_kernel<float><<<grid, block, 0, st>>>(a);
  else sample_faces_kernel<double><<<grid, block, 0, st>>>(a);
  pde::count_launch(1);
  return cudaGetLastError() == cudaSuccess ? PDE_OK : PDE_ERR_CUDA;
}

int pde_adam_step(const pde_adam* cfg, const void* grad_flat, void* exp_avg, void* exp_avg_sq, void* step,
                  void* stream) {
  if (!cfg || !grad_flat || !exp_avg || !exp_avg_sq || !step) return PDE_ERR_INVALID;
  if (cfg->dtype != PDE_F32 && cfg->dtype != PDE_F64) return PDE_ERR_INVALID;
  if (cfg->n_tensors < 1 || cfg->n_tensors > 2 * PDE_MAX_LINEAR + 1) return PDE_ERR_UNSUPPORTED;
  AdamArgs a;
  a.n_tensors = cfg->n_tensors;
  long long tot = 0;
  for (int i = 0; i < cfg->n_tensors; ++i) {
    if (!cfg->param[i] || cfg->numel[i] < 1) return PDE_ERR_INVALID;
    a.param[i] = cfg->param[i];
    a.start[i] = tot;
    tot += cfg->numel[i];
  }
  a.start[cfg->n_tensors] = tot;
  a.lr = cfg->lr; a.beta1 = cfg->beta1; a.beta2 = cfg->beta2; a.eps = cfg->eps; a.weight_decay = cfg->weight_decay;
  a.grad_scale = cfg->grad_scale;
  a.grad = grad_flat; a.m = exp_avg; a.v = exp_avg_sq; a.step = static_cast<const long long*>(step);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int block = 256, grid = grid_for(tot, block);
  if (cfg->dtype == PDE_F32) adam_kernel<float><<<grid, block, 0, st>>>(a);
  else adam_kernel<double><<<grid, block, 0, st>>>(a);
  if (cudaGetLastError() != cudaSuccess) return PDE_ERR_CUDA;
  bump_step_kernel<<<1, 1, 0, st>>>(static_cast<long long*>(step));
  pde::count_launch(2);
  return cudaGetLastError() == cudaSuccess ? PDE_OK : PDE_ERR_CUDA;
}

int pde_keep_best(const pde_adam* cfg, const void* metric, void* best_metric, void* best_flat, const void* step,
                  void* best_step, void* stream) {
  if (!cfg || !metric || !best_metric || !best_flat) return PDE_ERR_INVALID;
  if (cfg->dtype != PDE_F32 && cfg->dtype != PDE_F64) return PDE_ERR_INVALID;
  if (cfg->n_tensors < 1 || cfg->n_tensors > 2 * PDE_MAX_LINEAR + 1) return PDE_ERR_UNSUPPORTED;
  BestArgs a;
  a.n_tensors = cfg->n_tensors;
  long long tot = 0;
  for (int i = 0; i < cfg->n_tensors; ++i) {
    if (!cfg->param[i] || cfg->numel[i] < 1) return PDE_ERR_INVALID;
    a.param[i] = cfg->param[i];
    a.start[i] = tot;
    tot += cfg->numel[i];
  }
  a.start[cfg->n_tensors] = tot;
  a.metric = metric; a.best_metric = best_metric; a.best_flat = best_flat;
  a.step = static_cast<const long long*>(step); a.best_step = static_cast<long long*>(best_step);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (cfg->dtype == PDE_F32) keep_best_kernel<float><<<1, 1024, 0, st>>>(a);
  else keep_best_kernel<double><<<1, 1024, 0, st>>>(a);
  pde::count_launch(1);
  return cudaGetLastError() == cudaSuccess ? PDE_OK : PDE_ERR_CUDA;
}

}  // extern "C"
