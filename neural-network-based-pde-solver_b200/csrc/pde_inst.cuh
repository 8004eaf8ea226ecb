// pde_inst.cuh — explicit instantiation of the kernels for one floating-point type.
#pragma once
#include "pde_launch.h"

namespace pde {

template <typename T, int D, int ORDER>
static KernelInfo info_one() {
  cudaFuncAttributes at;
  KernelInfo k{reinterpret_cast<const void*>(&net_kernel<T, D, ORDER>), 255, 0};
  if (cudaFuncGetAttributes(&at, net_kernel<T, D, ORDER>) == cudaSuccess) {
    k.regs = at.numRegs;
    k.max_threads = at.maxThreadsPerBlock;
  } else {
    cudaGetLastError();
  }
  return k;
}

#define PDE_DISPATCH(T, dim, order, ...)                                       \
  switch ((dim) * 3 + (order)) {                                                \
    case 3:  { constexpr int D = 1, O = 0; __VA_ARGS__; } break;                       \
    case 4:  { constexpr int D = 1, O = 1; __VA_ARGS__; } break;                       \
    case 5:  { constexpr int D = 1, O = 2; __VA_ARGS__; } break;                       \
    case 6:  { constexpr int D = 2, O = 0; __VA_ARGS__; } break;                       \
    case 7:  { constexpr int D = 2, O = 1; __VA_ARGS__; } break;                       \
    case 8:  { constexpr int D = 2, O = 2; __VA_ARGS__; } break;                       \
    case 9:  { constexpr int D = 3, O = 0; __VA_ARGS__; } break;                       \
    case 10: { constexpr int D = 3, O = 1; __VA_ARGS__; } break;                       \
    case 11: { constexpr int D = 3, O = 2; __VA_ARGS__; } break;                       \
    case 12: { constexpr int D = 4, O = 0; __VA_ARGS__; } break;                       \
    case 13: { constexpr int D = 4, O = 1; __VA_ARGS__; } break;                       \
    case 14: { constexpr int D = 4, O = 2; __VA_ARGS__; } break;                       \
    case 15: { constexpr int D = 5, O = 0; __VA_ARGS__; } break;                       \
    case 16: { constexpr int D = 5, O = 1; __VA_ARGS__; } break;                       \
    case 17: { constexpr int D = 5, O = 2; __VA_ARGS__; } break;                       \
    default: break;                                                             \
  }

template <typename T>
static KernelInfo net_kernel_info_impl(int dim, int order) {
  KernelInfo k{nullptr, 0, 0};
  if (dim < 1 || dim > 5 || order < 0 || order > 2) return k;
  PDE_DISPATCH(T, dim, order, (k = info_one<T, D, O>()));
  return k;
}

template <typename T>
static cudaError_t launch_net_impl(int dim, int order, int grid, int block, size_t smem, cudaStream_t st,
                                   const KArgs<T>& a) {
  if (dim < 1 || dim > 5 || order < 0 || order > 2) return cudaErrorInvalidValue;
  cudaError_t err = cudaSuccess;
  PDE_DISPATCH(T, dim, order, {
    err = cudaFuncSetAttribute(net_kernel<T, D, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err == cudaSuccess) {
      net_kernel<T, D, O><<<grid, block, smem, st>>>(a);
      err = cudaGetLastError();
      count_launch();
    }
  });
  return err;
}

// ---- WAN pointwise kernel (oracle/jets_numpy.py: wan_means, bump_weight)
template <typename T>
__global__ void wan_kernel(const WanArgs<T> a) {
  const int D = a.D;
  double acc[5] = {0, 0, 0, 0, 0};
  for (long long gp = blockIdx.x * (long long)blockDim.x + threadIdx.x; gp < a.n;
       gp += (long long)gridDim.x * blockDim.x) {
    T x[5], bu[5], bu1[5], bv[5], bv1[5], tmp;
    for (int i = 0; i < D; ++i) {
      x[i] = a.X[gp * D + i];
      envelope_factor<T>(a.env_u, i, x[i], bu[i], bu1[i], tmp);
      envelope_factor<T>(a.env_v, i, x[i], bv[i], bv1[i], tmp);
    }
    // bump weight and its gradient
    const T h = (a.w_hi - a.w_lo) / T(2), cen = (a.w_hi + a.w_lo) / T(2);
    T ph[5], dph[5];
    for (int i = 0; i < D; ++i) {
      T t = (x[i] - cen) / h;
      if (fabs(t) < T(1)) {
        T den = t * t - T(1) + a.eps_den;
        ph[i] = exp_(T(1) / den) / T(0.210987);
        dph[i] = ph[i] * (T(-2) * t) / (den * den) / h;
      } else {
        ph[i] = T(0); dph[i] = T(0);
      }
    }
    T w = T(1), Bu = T(1), Bv = T(1);
    for (int i = 0; i < D; ++i) { w *= ph[i]; Bu *= bu[i]; Bv *= bv[i]; }
    T dw[5], Bui[5], Bvi[5];
    for (int i = 0; i < D; ++i) {
      T e = T(1), eu = T(1), ev = T(1);
      for (int j = 0; j < D; ++j)
        if (j != i) { e *= ph[j]; eu *= bu[j]; ev *= bv[j]; }
      dw[i] = dph[i] * e; Bui[i] = bu1[i] * eu; Bvi[i] = bv1[i] * ev;
    }
    const int C = 1 + D;
    const T Nu = a.Ju[gp * C], Nv = a.Jv[gp * C];
    const T u = Bu * Nu, v = Bv * Nv;
    T gu[5], gv[5], gphi[5];
    const T phi = w * v;
    for (int i = 0; i < D; ++i) {
      gu[i] = Bui[i] * Nu + Bu * a.Ju[gp * C + 1 + i];
      gv[i] = Bvi[i] * Nv + Bv * a.Jv[gp * C + 1 + i];
      gphi[i] = dw[i] * v + w * gv[i];
    }
    const T fv = a.f ? a.f[gp] : T(0);
    const T bt = a.beta ? a.beta[gp] : a.beta_const;
    const T E = a.energy ? a.energy[0] : a.energy_const;
    T dot = T(0), gv2 = T(0);
    for (int i = 0; i < D; ++i) { dot += gu[i] * gphi[i]; gv2 += gv[i] * gv[i]; }
    acc[0] += (double)(a.alpha * dot + (bt - E) * u * phi - fv * phi);
    acc[1] += (double)(phi * phi);
    acc[2] += (double)(u * u);
    acc[3] += (double)(gv2 + v * v);
    acc[4] += (double)(-u * phi);
    if (a.Jbar_u || a.Jbar_v) {
      T s[4];
      for (int k = 0; k < 4; ++k) s[k] = (a.seed ? a.seed[k] : T(1)) * a.inv_n;
      if (a.Jbar_u) {
        T ub = (bt - E) * phi * s[0] + T(2) * u * s[2];
        T n0 = Bu * ub;
        for (int i = 0; i < D; ++i) {
          T uib = a.alpha * gphi[i] * s[0];
          n0 += Bui[i] * uib;
          a.Jbar_u[gp * C + 1 + i] = Bu * uib;
        }
        a.Jbar_u[gp * C] = n0;
      }
      if (a.Jbar_v) {
        T dq_dphi = (bt - E) * u - fv;
        T vb = dq_dphi * w * s[0] + T(2) * phi * w * s[1] + T(2) * v * s[3];
        T n0;
        for (int i = 0; i < D; ++i) vb += a.alpha * gu[i] * dw[i] * s[0];
        n0 = Bv * vb;
        for (int i = 0; i < D; ++i) {
          T vib = a.alpha * gu[i] * w * s[0] + T(2) * gv[i] * s[3];
          n0 += Bvi[i] * vib;
          a.Jbar_v[gp * C + 1 + i] = Bv * vib;
        }
        a.Jbar_v[gp * C] = n0;
      }
    }
  }
  // block reduction in fixed order: warp shuffles then one thread over the warps
  __shared__ double sh[32][5];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    double v = acc[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) sh[wid][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    double v = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) v += sh[i][threadIdx.x];
    a.psums[(long long)blockIdx.x * 8 + threadIdx.x] = v;
  }
}

template <typename T>
__global__ void wan_finish_kernel(const double* psums, int blocks, T* sums) {
  if (threadIdx.x < 5) {
    double v = 0.0;
    for (int b = 0; b < blocks; ++b) v += psums[(long long)b * 8 + threadIdx.x];
    sums[threadIdx.x] = (T)v;
  }
}

template <typename T>
static cudaError_t launch_wan_impl(cudaStream_t st, const WanArgs<T>& a) {
  wan_kernel<T><<<a.blocks, 256, 0, st>>>(a);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return err;
  wan_finish_kernel<T><<<1, 32, 0, st>>>(a.psums, a.blocks, a.sums);
  count_launch(2);
  return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_pack_impl(cudaStream_t st, const PackArgs<T>& a) {
  int blocks = (int)((a.total + 255) / 256);
  if (blocks > 1184) blocks = 1184;
  pack_kernel<T><<<blocks, 256, 0, st>>>(a);
  count_launch();
  return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_reduce_impl(cudaStream_t st, const ReduceArgs<T>& a) {
  long long total = a.n_params + a.n_q + 1;
  int blocks = (int)((total + 127) / 128);
  reduce_kernel<T><<<blocks, 128, 0, st>>>(a);
  count_launch();
  return cudaGetLastError();
}

#define PDE_INSTANTIATE(T)                                                                              \
  template <> KernelInfo net_kernel_info<T>(int dim, int order) { return net_kernel_info_impl<T>(dim, order); } \
  template <> cudaError_t launch_net<T>(int dim, int order, int grid, int block, size_t smem, cudaStream_t st,   \
                                        const KArgs<T>& a) {                                            \
    return launch_net_impl<T>(dim, order, grid, block, smem, st, a);                                    \
  }                                                                                                     \
  template <> cudaError_t launch_pack<T>(cudaStream_t st, const PackArgs<T>& a) { return launch_pack_impl<T>(st, a); } \
  template <> cudaError_t launch_reduce<T>(cudaStream_t st, const ReduceArgs<T>& a) { return launch_reduce_impl<T>(st, a); } \
  template <> cudaError_t launch_wan<T>(cudaStream_t st, const WanArgs<T>& a) { return launch_wan_impl<T>(st, a); }

}  // namespace pde
