// pde_simt.cuh — generic fused collocation kernel (SIMT FMA path, fp32 and fp64).
//
// One CTA owns a tile of P points.  Thread (p, ug) owns the micro-tile "all C jet channels x
// 4 hidden units" of point p, so the sin/tanh chain rule (which mixes the channels of one
// (point, unit)) is thread local.  Per tile, entirely in shared memory:
//   forward : layer 0 from x, hidden layers as register-tiled GEMMs (activations broadcast
//             from smem, weights streamed global->smem in K chunks), pre-activations stashed;
//   program : envelope + residual + per-point seeds (or jets out / cotangents in);
//   reverse : dgrad GEMMs, activation adjoints in place over the stash, wgrad micro-tiles
//             accumulated into this CTA's private partial-gradient vector in global memory.
// A second kernel sums the per-CTA partials in fixed order (deterministic).
//
// What it computes follows the reference's nested-autograd path:
//   Poisson_Equations/Poisson_ND.py:11-33 (network, envelope), :61-71 (grad, Laplacian),
//   :91-103 (PINN / Deep-Ritz losses), :240 (loss.backward()).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "pde_comm.cuh"

namespace pde {

enum Mode { MODE_JETS_FWD = 0, MODE_JETS_BWD = 1, MODE_PROGRAM = 2 };

// separable envelope description (pde_envelope in include/pde_b200.h)
template <typename T>
struct EnvDev {
  int kind;
  int n_nodes[5];
  T nodes[5][8];
  T lo, hi;
};

template <typename T>
struct KArgs {
  // network geometry
  int n_h, H, Hp, UG, act;
  int P, KC, pitchP;
  // packed parameters (element offsets into `packed`)
  const T* packed;
  long long off_W0t, off_b, off_Wt, off_Wn, off_wL, off_bL;
  // points
  const T* X;
  long long n;
  int num_tiles;
  // mode / io
  int mode, want_grad;
  T* J;
  const T* Jbar;
  // program
  int prog, n_q;
  EnvDev<T> env;
  T alpha, beta_const, energy_const, inv_n;
  const T* f;
  const T* beta;
  const T* energy;
  const T* seed;
  // per-CTA partial vectors (gradients in T, q sums in double: psums[cta][8] = q0..q3, dq/dE)
  T* partial;
  double* psums;
  long long PP, off_gW0, off_gb0, off_gW, off_gwL, off_gbL;
  // PDE_PROG_FLUX: face mask and points per face (n / popcount(faces))
  int faces;
  long long face_n;
};

// Outward normal of the face that point gp of a PDE_PROG_FLUX batch lies on (include/pde_b200.h: one block of face_n
// points per set bit of `faces`, in increasing bit order): axis in [0, dim), sign -1 (lo face) or +1 (hi face).
// A subtraction walk over at most 2*dim - 1 blocks instead of a 64-bit division.
__device__ __forceinline__ void flux_face(int faces, long long face_n, long long gp, int& axis, int& sign) {
  unsigned m = (unsigned)faces;
  for (long long r = gp; r >= face_n; r -= face_n) m &= m - 1u;
  const int k = __ffs((int)m) - 1;
  axis = k >> 1;
  sign = (k & 1) ? 1 : -1;
}

// ---------------------------------------------------------------- small helpers
template <typename T> __device__ __forceinline__ void ld4(const T* p, T (&v)[4]);
template <> __device__ __forceinline__ void ld4<float>(const float* p, float (&v)[4]) {
  float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <> __device__ __forceinline__ void ld4<double>(const double* p, double (&v)[4]) {
  double2 a = *reinterpret_cast<const double2*>(p);
  double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
template <typename T> __device__ __forceinline__ void st4(T* p, const T (&v)[4]);
template <> __device__ __forceinline__ void st4<float>(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <> __device__ __forceinline__ void st4<double>(double* p, const double (&v)[4]) {
  *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
  *reinterpret_cast<double2*>(p + 2) = make_double2(v[2], v[3]);
}

__device__ __forceinline__ void sincos_(float z, float* s, float* c) { sincosf(z, s, c); }
__device__ __forceinline__ void sincos_(double z, double* s, double* c) { sincos(z, s, c); }
__device__ __forceinline__ float tanh_(float z) { return tanhf(z); }
__device__ __forceinline__ double tanh_(double z) { return tanh(z); }
__device__ __forceinline__ float exp_(float z) { return expf(z); }
__device__ __forceinline__ double exp_(double z) { return exp(z); }

// sigma and its first three derivatives (sin: Poisson_ND.py:8-9; tanh: IPW_1D_WAN.py:71)
template <typename T>
__device__ __forceinline__ void act_derivs(int act, T z, T& s0, T& s1, T& s2, T& s3) {
  if (act == 0) {
    T s, c;
    sincos_(z, &s, &c);
    s0 = s; s1 = c; s2 = -s; s3 = -c;
  } else {
    T t = tanh_(z);
    T d1 = T(1) - t * t;
    s0 = t; s1 = d1; s2 = T(-2) * t * d1; s3 = T(-2) * d1 * (T(1) - T(3) * t * t);
  }
}

// ---------------------------------------------------------------- shared-memory carve-up
template <typename T, int C>
struct Smem {
  T* W0t;   // [D][Hp]
  T* B;     // [n_h][Hp]
  T* wL;    // [Hp] (+1: bL)
  T* X;     // [P][D]
  T* out;   // [P][C]
  T* red;   // [P][C][UG]
  T* A;     // [P][pitchP]
  T* Z;     // [n_h][P][pitchP]
  T* Wc;    // [KC][Hp]
};

__host__ __device__ inline long long align4(long long x) { return (x + 3) & ~3LL; }

template <typename T>
__host__ __device__ inline long long smem_elems(int D, int C, int n_h, int Hp, int UG, int P, int KC, int pitchP) {
  long long e = 0;
  e += align4((long long)D * Hp);
  e += align4((long long)n_h * Hp);
  e += align4(Hp + 4);
  e += align4((long long)P * D);
  e += align4((long long)P * C);
  e += align4((long long)P * C * UG + 5LL * P);
  e += align4((long long)P * pitchP);
  e += align4((long long)n_h * P * pitchP);
  e += align4((long long)KC * Hp);
  return e;
}

// ---------------------------------------------------------------- register-tiled GEMM
// acc[c][u] += sum_k In[p][c][k] * Wg[k][4*ug+u],   k in [0,Hp);  Wg is a global [Hp][Hp] matrix
// streamed through the smem chunk buffer Wc.  Used for the forward (Wg = W^T) and for dgrad
// (Wg = W, natural layout).
template <typename T, int C>
__device__ __forceinline__ void gemm_tile(const KArgs<T>& a, const T* __restrict__ Wg, const T* sIn,
                                          T* sWc, int p, int ug, T (&acc)[C][4]) {
  const int Hp = a.Hp, KC = a.KC;
  const T* in_p = sIn + (long long)p * a.pitchP;
  for (int k0 = 0; k0 < Hp; k0 += KC) {
    const int kc = min(KC, Hp - k0);
    __syncthreads();  // previous users of Wc are done
    {
      const int n4 = (kc * Hp) >> 2;
      const T* src = Wg + (long long)k0 * Hp;
      for (int i = threadIdx.x; i < n4; i += blockDim.x) {
        T v[4];
        ld4<T>(src + 4 * i, v);
        st4<T>(sWc + 4 * i, v);
      }
    }
    __syncthreads();
#pragma unroll 1
    for (int k = 0; k < kc; k += 4) {
      T av[C][4];
#pragma unroll
      for (int c = 0; c < C; ++c) ld4<T>(in_p + c * Hp + k0 + k, av[c]);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        T w[4];
        ld4<T>(sWc + (k + kk) * Hp + 4 * ug, w);
#pragma unroll
        for (int c = 0; c < C; ++c) {
#pragma unroll
          for (int u = 0; u < 4; ++u) acc[c][u] = fma(av[c][kk], w[u], acc[c][u]);
        }
      }
    }
  }
}

// ---------------------------------------------------------------- envelope factor b(t), b'(t), b''(t)
// (oracle/jets_numpy.py: envelope_factors; Poisson_ND.py:28, QHO_2D.py:151-168)
template <typename T>
__device__ __forceinline__ void envelope_factor(const EnvDev<T>& e, int i, T t, T& b, T& b1, T& b2) {
  if (e.kind == 1) {
    b = (t - e.lo) * (e.hi - t); b1 = (e.lo + e.hi) - T(2) * t; b2 = T(-2);
  } else if (e.kind == 2) {
    T pp = exp_(-(t - e.lo)), qq = exp_(t - e.hi);
    b = (T(1) - pp) * (T(1) - qq);
    b1 = pp * (T(1) - qq) - (T(1) - pp) * qq;
    b2 = -pp * (T(1) - qq) - T(2) * pp * qq - (T(1) - pp) * qq;
  } else {
    b = T(1); b1 = T(0); b2 = T(0);
  }
  for (int k = 0; k < e.n_nodes[i]; ++k) {
    T g = t - e.nodes[i][k];
    b2 = b2 * g + T(2) * b1;
    b1 = b1 * g + b;
    b = b * g;
  }
}

// ---------------------------------------------------------------- envelope + residual program
// Per point: network jets nj[C] -> q sums and cotangents nb[C] of the network jets.
template <typename T, int D, int ORDER>
__device__ void program_point(const KArgs<T>& a, const T* x, long long gp, T (&nj)[1 + ORDER * D],
                              double (&qs)[4], double& gE) {
  T b[D], b1[D], b2[D];
#pragma unroll
  for (int i = 0; i < D; ++i) envelope_factor<T>(a.env, i, x[i], b[i], b1[i], b2[i]);
  T B = T(1);
#pragma unroll
  for (int i = 0; i < D; ++i) B *= b[i];
  T Bi[D], Bii[D];
#pragma unroll
  for (int i = 0; i < D; ++i) {
    T e = T(1);
#pragma unroll
    for (int j = 0; j < D; ++j)
      if (j != i) e *= b[j];
    Bi[i] = b1[i] * e; Bii[i] = b2[i] * e;
  }
  // u jets
  const T N0 = nj[0];
  T u = B * N0, ui[D], uii[D];
#pragma unroll
  for (int i = 0; i < D; ++i) {
    ui[i] = T(0); uii[i] = T(0);
    if constexpr (ORDER >= 1) ui[i] = Bi[i] * N0 + B * nj[1 + i];
    if constexpr (ORDER >= 2) uii[i] = Bii[i] * N0 + T(2) * Bi[i] * nj[1 + i] + B * nj[1 + D + i];
  }
  const T fv = a.f ? a.f[gp] : T(0);
  const T bt = a.beta ? a.beta[gp] : a.beta_const;
  const T E = a.energy ? a.energy[0] : a.energy_const;
  const T w0 = (a.seed ? a.seed[0] : T(1)) * a.inv_n;
  T ub = T(0), uib[D], uiib[D];
#pragma unroll
  for (int i = 0; i < D; ++i) { uib[i] = T(0); uiib[i] = T(0); }
  if (a.prog == 1) {  // PINN
    T lap = T(0);
#pragma unroll
    for (int i = 0; i < D; ++i) lap += uii[i];
    T r = a.alpha * lap + (bt - E) * u - fv;
    qs[0] += (double)(r * r);
    T rb = T(2) * r * w0;
    ub = (bt - E) * rb;
#pragma unroll
    for (int i = 0; i < D; ++i) uiib[i] = a.alpha * rb;
    gE += (double)(-u * rb);
  } else if (a.prog == 2) {  // Deep Ritz
    T g2 = T(0);
#pragma unroll
    for (int i = 0; i < D; ++i) g2 += ui[i] * ui[i];
    qs[0] += (double)(a.alpha * g2 - fv * u);
    ub = -fv * w0;
#pragma unroll
    for (int i = 0; i < D; ++i) uib[i] = T(2) * a.alpha * ui[i] * w0;
  } else if (a.prog == 3) {  // Rayleigh quotient pieces
    T g2 = T(0);
#pragma unroll
    for (int i = 0; i < D; ++i) g2 += ui[i] * ui[i];
    qs[0] += (double)(a.alpha * g2 + bt * u * u);
    qs[1] += (double)(u * u);
    const T w1 = (a.seed ? a.seed[1] : T(1)) * a.inv_n;
    ub = T(2) * bt * u * w0 + T(2) * u * w1;
#pragma unroll
    for (int i = 0; i < D; ++i) uib[i] = T(2) * a.alpha * ui[i] * w0;
  } else if (ORDER == 1 && a.prog == 5) {  // boundary flux: r = alpha n.grad u + beta u - g
    int ax, sg;
    flux_face(a.faces, a.face_n, gp, ax, sg);
    const T as = sg > 0 ? a.alpha : -a.alpha;
    T un = T(0);
#pragma unroll
    for (int i = 0; i < D; ++i)
      if (i == ax) un = ui[i];
    const T r = as * un + bt * u - fv;
    qs[0] += (double)(r * r);
    const T rb = T(2) * r * w0;
    ub = bt * rb;
#pragma unroll
    for (int i = 0; i < D; ++i) uib[i] = (i == ax) ? as * rb : T(0);
  } else {  // MSE on the value
    T r = u - fv;
    qs[0] += (double)(r * r);
    ub = T(2) * r * w0;
  }
  // envelope adjoint
  T n0b = B * ub;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    if constexpr (ORDER >= 1) {
      n0b += Bi[i] * uib[i];
      T t1 = B * uib[i];
      if constexpr (ORDER >= 2) {
        n0b += Bii[i] * uiib[i];
        t1 += T(2) * Bi[i] * uiib[i];
        nj[1 + D + i] = B * uiib[i];
      }
      nj[1 + i] = t1;
    }
  }
  nj[0] = n0b;
}

// ---------------------------------------------------------------- the kernel
template <typename T, int D, int ORDER>
__global__ void net_kernel(const KArgs<T> a) {
  constexpr int C = 1 + ORDER * D;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  const int Hp = a.Hp, UG = a.UG, P = a.P, n_h = a.n_h, pitchP = a.pitchP;
  Smem<T, C> s;
  s.W0t = sp; sp += align4((long long)D * Hp);
  s.B = sp;   sp += align4((long long)n_h * Hp);
  s.wL = sp;  sp += align4(Hp + 4);
  s.X = sp;   sp += align4((long long)P * D);
  s.out = sp; sp += align4((long long)P * C);
  s.red = sp; sp += align4((long long)P * C * UG + 5LL * P);
  s.A = sp;   sp += align4((long long)P * pitchP);
  s.Z = sp;   sp += align4((long long)n_h * P * pitchP);
  s.Wc = sp;

  const int tid = threadIdx.x, nt = blockDim.x;
  const int p = tid / UG, ug = tid % UG;
  const bool do_bwd = (a.mode == MODE_JETS_BWD) || (a.mode == MODE_PROGRAM && a.want_grad);
  T* part = a.partial + (long long)blockIdx.x * a.PP;

  // persistent small parameters; zero this CTA's partial vector
  for (int i = tid; i < D * Hp; i += nt) s.W0t[i] = a.packed[a.off_W0t + i];
  for (int i = tid; i < n_h * Hp; i += nt) s.B[i] = a.packed[a.off_b + i];
  for (int i = tid; i < Hp; i += nt) s.wL[i] = a.packed[a.off_wL + i];
  if (tid == 0) s.wL[Hp] = a.packed[a.off_bL];
  if (do_bwd)
    for (long long i = tid; i < a.PP; i += nt) part[i] = T(0);
  double qs[4] = {0.0, 0.0, 0.0, 0.0};  // sums of q in double whatever T is
  double gE = 0.0;
  __syncthreads();

  for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x) {
    const long long base = (long long)tile * P;
    // ---- points of this tile (padded points replicate nothing: x = 0, seeds = 0)
    for (int i = tid; i < P * D; i += nt) {
      long long gp = base + i / D;
      s.X[i] = (gp < a.n) ? a.X[gp * D + (i % D)] : T(0);
    }
    __syncthreads();

    // ---- layer 0: z = W0 x + b0, z'_j = W0[:,j], z''_j = 0
    {
      T z[C][4];
      T xv[D];
#pragma unroll
      for (int j = 0; j < D; ++j) xv[j] = s.X[p * D + j];
      T bb[4];
      ld4<T>(s.B + 4 * ug, bb);
#pragma unroll
      for (int u = 0; u < 4; ++u) z[0][u] = bb[u];
#pragma unroll
      for (int j = 0; j < D; ++j) {
        T w[4];
        ld4<T>(s.W0t + j * Hp + 4 * ug, w);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          z[0][u] = fma(w[u], xv[j], z[0][u]);
          if constexpr (ORDER >= 1) z[1 + j][u] = w[u];
          if constexpr (ORDER >= 2) z[1 + D + j][u] = T(0);
        }
      }
      T* zrow = s.Z + (long long)p * pitchP + 4 * ug;
      T* arow = s.A + (long long)p * pitchP + 4 * ug;
      T av[C][4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        T s0, s1, s2, s3;
        act_derivs<T>(a.act, z[0][u], s0, s1, s2, s3);
        av[0][u] = s0;
#pragma unroll
        for (int i = 0; i < D; ++i) {
          if constexpr (ORDER >= 1) av[1 + i][u] = s1 * z[1 + i][u];
          if constexpr (ORDER >= 2) av[1 + D + i][u] = s2 * z[1 + i][u] * z[1 + i][u];
        }
      }
#pragma unroll
      for (int c = 0; c < C; ++c) {
        st4<T>(zrow + c * Hp, z[c]);
        st4<T>(arow + c * Hp, av[c]);
      }
    }
    __syncthreads();

    // ---- hidden layers 1..n_h-1
    T alast[C][4];  // activations of the last hidden layer (kept for the output layer)
    for (int l = 1; l < n_h; ++l) {
      T acc[C][4];
      {
        T bb[4];
        ld4<T>(s.B + l * Hp + 4 * ug, bb);
#pragma unroll
        for (int c = 0; c < C; ++c)
#pragma unroll
          for (int u = 0; u < 4; ++u) acc[c][u] = (c == 0) ? bb[u] : T(0);
      }
      gemm_tile<T, C>(a, a.packed + a.off_Wt + (long long)(l - 1) * Hp * Hp, s.A, s.Wc, p, ug, acc);
      __syncthreads();  // everyone finished reading A
      T* zrow = s.Z + ((long long)l * P + p) * pitchP + 4 * ug;
      T* arow = s.A + (long long)p * pitchP + 4 * ug;
#pragma unroll
      for (int c = 0; c < C; ++c) st4<T>(zrow + c * Hp, acc[c]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        T s0, s1, s2, s3;
        act_derivs<T>(a.act, acc[0][u], s0, s1, s2, s3);
        alast[0][u] = s0;
#pragma unroll
        for (int i = 0; i < D; ++i) {
          if constexpr (ORDER >= 1) alast[1 + i][u] = s1 * acc[1 + i][u];
          if constexpr (ORDER >= 2) alast[1 + D + i][u] = s2 * acc[1 + i][u] * acc[1 + i][u] + s1 * acc[1 + D + i][u];
        }
      }
#pragma unroll
      for (int c = 0; c < C; ++c) st4<T>(arow + c * Hp, alast[c]);
      __syncthreads();
    }
    if (n_h == 1) {
      const T* arow = s.A + (long long)p * pitchP + 4 * ug;
#pragma unroll
      for (int c = 0; c < C; ++c) ld4<T>(arow + c * Hp, alast[c]);
    }

    // ---- output layer (width 1): N_c = wL . a_c (+ bL)
    {
      T w[4];
      ld4<T>(s.wL + 4 * ug, w);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        T v = T(0);
#pragma unroll
        for (int u = 0; u < 4; ++u) v = fma(w[u], alast[c][u], v);
        s.red[((long long)p * C + c) * UG + ug] = v;
      }
    }
    __syncthreads();
    for (int i = tid; i < P * C; i += nt) {
      T v = (i % C == 0) ? s.wL[Hp] : T(0);
      const T* r = s.red + (long long)i * UG;
      for (int g = 0; g < UG; ++g) v += r[g];
      s.out[i] = v;
    }
    __syncthreads();

    // ---- jets out / program / cotangents in
    if (a.mode == MODE_JETS_FWD) {
      for (int i = tid; i < P * C; i += nt) {
        long long gp = base + i / C;
        if (gp < a.n) a.J[gp * C + (i % C)] = s.out[i];
      }
    } else if (a.mode == MODE_JETS_BWD) {
      for (int i = tid; i < P * C; i += nt) {
        long long gp = base + i / C;
        s.out[i] = (gp < a.n) ? a.Jbar[gp * C + (i % C)] : T(0);
      }
    } else {
      if (tid < P) {
        long long gp = base + tid;
        T nj[C];
#pragma unroll
        for (int c = 0; c < C; ++c) nj[c] = s.out[tid * C + c];
        if (gp < a.n) {
          program_point<T, D, ORDER>(a, s.X + tid * D, gp, nj, qs, gE);
        } else {
#pragma unroll
          for (int c = 0; c < C; ++c) nj[c] = T(0);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) s.out[tid * C + c] = nj[c];
      }
    }
    __syncthreads();
    if (!do_bwd) continue;

    // ---- reverse sweep
    for (int l = n_h - 1; l >= 0; --l) {
      T ab[C][4];
      if (l == n_h - 1) {
        T w[4];
        ld4<T>(s.wL + 4 * ug, w);
#pragma unroll
        for (int c = 0; c < C; ++c) {
          T nb = s.out[p * C + c];
#pragma unroll
          for (int u = 0; u < 4; ++u) ab[c][u] = w[u] * nb;
        }
      } else {
#pragma unroll
        for (int c = 0; c < C; ++c)
#pragma unroll
          for (int u = 0; u < 4; ++u) ab[c][u] = T(0);
        gemm_tile<T, C>(a, a.packed + a.off_Wn + (long long)l * Hp * Hp, s.Z + (long long)(l + 1) * P * pitchP,
                        s.Wc, p, ug, ab);
      }
      // activation adjoint of layer l, in place over the stash; recompute A_l into s.A
      {
        T* zrow = s.Z + ((long long)l * P + p) * pitchP + 4 * ug;
        T* arow = s.A + (long long)p * pitchP + 4 * ug;
        T z[C][4];
#pragma unroll
        for (int c = 0; c < C; ++c) ld4<T>(zrow + c * Hp, z[c]);
        T zb[C][4], av[C][4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          T s0, s1, s2, s3;
          act_derivs<T>(a.act, z[0][u], s0, s1, s2, s3);
          av[0][u] = s0;
          T zb0 = s1 * ab[0][u];
#pragma unroll
          for (int i = 0; i < D; ++i) {
            if constexpr (ORDER >= 1) {
              const T z1 = z[1 + i][u], ab1 = ab[1 + i][u];
              av[1 + i][u] = s1 * z1;
              zb0 = fma(s2 * z1, ab1, zb0);
              T t1 = s1 * ab1;
              if constexpr (ORDER >= 2) {
                const T z2 = z[1 + D + i][u], ab2 = ab[1 + D + i][u];
                av[1 + D + i][u] = s2 * z1 * z1 + s1 * z2;
                zb0 = fma(s3 * z1 * z1 + s2 * z2, ab2, zb0);
                t1 = fma(T(2) * s2 * z1, ab2, t1);
                zb[1 + D + i][u] = s1 * ab2;
              }
              zb[1 + i][u] = t1;
            }
          }
          zb[0][u] = zb0;
        }
        // the dgrad GEMM above read Z[l+1] and (for l<n_h-1) nothing of Z[l]/A, so in-place is safe
#pragma unroll
        for (int c = 0; c < C; ++c) {
          st4<T>(zrow + c * Hp, zb[c]);
          st4<T>(arow + c * Hp, av[c]);
        }
      }
      __syncthreads();
      // parameter gradients that pair Zbar_{l+1} (or the output cotangent) with A_l
      if (l == n_h - 1) {
        for (int uo = tid; uo < Hp; uo += nt) {
          T g = T(0);
          for (int pp = 0; pp < P; ++pp)
            for (int c = 0; c < C; ++c) g = fma(s.out[pp * C + c], s.A[(long long)pp * pitchP + c * Hp + uo], g);
          part[a.off_gwL + uo] += g;
        }
        if (tid == 0) {
          // bias gradients are plain sums of signed cotangents over the points (for WAN critics they cancel to a
          // small remainder): summed in double so that the result carries the rounding of the terms only
          double g = 0.0;
          for (int pp = 0; pp < P; ++pp) g += (double)s.out[pp * C];
          part[a.off_gbL] += (T)g;
        }
      } else {
        const T* Zb = s.Z + (long long)(l + 1) * P * pitchP;
        T* gW = part + a.off_gW + (long long)l * ((long long)Hp * Hp + Hp);  // layer l+1 lives at slot l
        for (int mt = tid; mt < UG * UG; mt += nt) {
          const int og = mt / UG, ig = mt % UG;
          T g[4][4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) g[i][j] = T(0);
          for (int pp = 0; pp < P; ++pp) {
            const T* zr = Zb + (long long)pp * pitchP + 4 * og;
            const T* ar = s.A + (long long)pp * pitchP + 4 * ig;
#pragma unroll
            for (int c = 0; c < C; ++c) {
              T zv[4], avv[4];
              ld4<T>(zr + c * Hp, zv);
              ld4<T>(ar + c * Hp, avv);
#pragma unroll
              for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) g[i][j] = fma(zv[i], avv[j], g[i][j]);
            }
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            T* dst = gW + (long long)(4 * og + i) * Hp + 4 * ig;
            T cur[4];
            ld4<T>(dst, cur);
#pragma unroll
            for (int j = 0; j < 4; ++j) cur[j] += g[i][j];
            st4<T>(dst, cur);
          }
        }
        T* gb = gW + (long long)Hp * Hp;
        for (int o = tid; o < Hp; o += nt) {
          double g = 0.0;
          for (int pp = 0; pp < P; ++pp) g += (double)Zb[(long long)pp * pitchP + o];
          gb[o] += (T)g;
        }
      }
      __syncthreads();
    }
    // layer 0 parameters from Zbar_0 and x
    for (int i = tid; i < Hp * D; i += nt) {
      const int o = i / D, j = i % D;
      T g = T(0);
      for (int pp = 0; pp < P; ++pp) {
        const T* zr = s.Z + (long long)pp * pitchP;
        g = fma(zr[o], s.X[pp * D + j], g);
        if constexpr (ORDER >= 1) g += zr[(1 + j) * Hp + o];
      }
      part[a.off_gW0 + i] += g;
    }
    for (int o = tid; o < Hp; o += nt) {
      double g = 0.0;
      for (int pp = 0; pp < P; ++pp) g += (double)s.Z[(long long)pp * pitchP + o];
      part[a.off_gb0 + o] += (T)g;
    }
    __syncthreads();
  }

  // per-CTA sums of q and dq/dE in fixed order
  if (a.mode == MODE_PROGRAM) {
    __syncthreads();
    double* dred = reinterpret_cast<double*>(s.A);  // P*5 doubles fit in the activation buffer
    if (tid < P) {
#pragma unroll
      for (int k = 0; k < 4; ++k) dred[tid * 5 + k] = qs[k];
      dred[tid * 5 + 4] = gE;
    }
    __syncthreads();
    for (int k = tid; k < 5; k += nt) {   // (a CTA can have fewer than 5 threads: tiny batches of narrow nets)
      double v = 0.0;
      for (int pp = 0; pp < P; ++pp) v += dred[pp * 5 + k];
      a.psums[(long long)blockIdx.x * 8 + k] = v;
    }
  }
}

// ---------------------------------------------------------------- parameter packing
template <typename T>
struct PackArgs {
  const T* W[8];
  const T* b[8];
  int n_lin, D, H, Hp;
  T* packed;
  long long off_W0t, off_b, off_Wt, off_Wn, off_wL, off_bL, total;
};

template <typename T>
__global__ void pack_kernel(const PackArgs<T> a) {
  const int n_h = a.n_lin - 1;
  const long long HH = (long long)a.Hp * a.Hp;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.total;
       i += (long long)gridDim.x * blockDim.x) {
    T v = T(0);
    if (i >= a.off_bL) {
      if (i == a.off_bL) v = a.b[n_h][0];
    } else if (i >= a.off_wL) {
      long long u = i - a.off_wL;
      if (u < a.H) v = a.W[n_h][u];
    } else if (i >= a.off_Wn) {
      long long r = i - a.off_Wn;
      int l = (int)(r / HH) + 1;  // slot l-1 holds W_l (natural layout)
      long long e = r % HH;
      int o = (int)(e / a.Hp), k = (int)(e % a.Hp);
      if (o < a.H && k < a.H) v = a.W[l][(long long)o * a.H + k];
    } else if (i >= a.off_Wt) {
      long long r = i - a.off_Wt;
      int l = (int)(r / HH) + 1;  // slot l-1 holds W_l^T
      long long e = r % HH;
      int k = (int)(e / a.Hp), o = (int)(e % a.Hp);
      if (o < a.H && k < a.H) v = a.W[l][(long long)o * a.H + k];
    } else if (i >= a.off_b) {
      long long r = i - a.off_b;
      int l = (int)(r / a.Hp), o = (int)(r % a.Hp);
      if (o < a.H) v = a.b[l][o];
    } else {
      long long r = i - a.off_W0t;
      int j = (int)(r / a.Hp), o = (int)(r % a.Hp);
      if (o < a.H) v = a.W[0][(long long)o * a.D + j];
    }
    a.packed[i] = v;
  }
}

// ---------------------------------------------------------------- fixed-order reduction of the per-CTA partials
template <typename T>
struct ReduceArgs {
  const T* partial;
  const double* psums;
  long long PP;
  int grid, n_lin, D, H, Hp, n_q;
  long long off_gW0, off_gb0, off_gW, off_gwL, off_gbL;
  long long n_params;
  T* grad;         // may be null
  T* sums;         // may be null
  T* energy_grad;  // may be null
  // Exchange fused into the reduction (pde_residual_loss_grad_exchange): every reduced element is pushed to the peers
  // and summed over the ranks before it is written; slot index = position in the caller's [grad | dE | sums] vector.
  int have_comm;
  comm::CommArgs comm;
  int psum_grid;    // rows of psums (0: same as grid) — the dimension-split PINN step takes them from its pointwise kernel
  int accumulate;   // add the reduced gradient to what grad already holds (second pass of that step)
};

template <typename T>
__global__ void reduce_kernel(const ReduceArgs<T> a) {
  const long long total = a.n_params + a.n_q + 1;
  const uint32_t call = a.have_comm ? *a.comm.seq + 1u : 0u;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long src = 0;
    T* dst;
    if (i >= a.n_params) {
      const int k = (int)(i - a.n_params);  // 0..n_q-1: q sums; n_q: dq/dE
      dst = (k < a.n_q) ? (a.sums ? a.sums + k : nullptr) : a.energy_grad;
      if (!dst) continue;
      const int col = (k < a.n_q) ? k : 4;
      double v = 0.0;
      const int pg = a.psum_grid > 0 ? a.psum_grid : a.grid;
#pragma unroll 8
      for (int g = 0; g < pg; ++g) v += a.psums[(long long)g * 8 + col];
      T r = (T)v;
      if (a.have_comm) r = comm::exchange_element<T>(a.comm, (k < a.n_q) ? a.n_params + 1 + k : a.n_params, r, call);
      *dst = r;
      continue;
    }
    {
      if (!a.grad) continue;
      dst = a.grad + i;
      // locate (layer, W|b, row, col) of flat index i
      long long r = i;
      const long long n0 = (long long)a.H * a.D + a.H;
      const long long nm = (long long)a.H * a.H + a.H;
      const int n_h = a.n_lin - 1;
      if (r < n0) {
        if (r < (long long)a.H * a.D) src = a.off_gW0 + r;  // [H][D] rows contiguous in both layouts
        else src = a.off_gb0 + (r - (long long)a.H * a.D);
      } else {
        r -= n0;
        int l = (int)(r / nm) + 1;
        if (l < n_h) {
          long long e = r % nm;
          long long slot = a.off_gW + (long long)(l - 1) * ((long long)a.Hp * a.Hp + a.Hp);
          if (e < (long long)a.H * a.H) src = slot + (e / a.H) * a.Hp + (e % a.H);
          else src = slot + (long long)a.Hp * a.Hp + (e - (long long)a.H * a.H);
        } else {
          long long e = r - (long long)(n_h - 1) * nm;
          src = (e < a.H) ? a.off_gwL + e : a.off_gbL;
        }
      }
    }
    // fixed order g = 0, 1, ...; unrolled so that 32 of the (independent, L2-latency) loads are in flight
    double v = 0.0;
#pragma unroll 32
    for (int g = 0; g < a.grid; ++g) v += (double)a.partial[(long long)g * a.PP + src];
    T r = (T)v;
    if (a.accumulate) r += *dst;
    if (a.have_comm) r = comm::exchange_element<T>(a.comm, i, r, call);
    *dst = r;
  }
  if (a.have_comm) comm::finish_call(a.comm, call);
}

}  // namespace pde
