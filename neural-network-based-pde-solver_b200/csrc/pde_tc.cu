// pde_tc.cu — Blackwell tensor-core (tcgen05 / TMEM) fused collocation loss step, fp32 parity
// through 3-term fp16 operand splits (x = hi + lo; hi*hi + lo*hi + hi*lo, fp32 accumulate).
//
// What it computes is the reference's nested-autograd step (Poisson_Equations/Poisson_ND.py:61-71
// grad / Laplacian, :91-103 PINN / Deep-Ritz losses, :240 loss.backward()) for networks
// [d, H<=64, ..., H, 1] with 2..4 hidden layers, restated as
//   * forward-mode jets with a *Laplacian* channel instead of d second-derivative channels:
//       channels (value, d_1..d_d, Lap):  z = W a (+b on the value channel),
//       a0 = s(z0),  a_i = s'(z0) z_i,  aL = s'(z0) zL + s''(z0) sum_i z_i^2,
//     which is the same quantity the reference sums from the Hessian diagonal (Poisson_ND.py:67-71);
//   * the reverse sweep of that recurrence, fused in the same pass over a tile of 64 points.
//
// One persistent CTA per SM walks 64-point tiles.  Per hidden GEMM layer the three contractions
//   forward  Z_c   = A_c   W^T      (M = 64 points, N = 64 units, K = 64 units)
//   dgrad    Ab_c  = Zb_c  W        (same shape, B operand = the same W tile viewed MN-major)
//   wgrad    gW   += Zb_c^T A_c     (M = N = 64 units, K = 64 points, both operands MN-major views)
// are tcgen05.mma kind::f16 instructions with accumulators in TMEM (forward / dgrad: two channels stacked along
// M = 128 per instruction, see ch_paired; wgrad: M = 64); the sin/tanh chain rule, the fp16 hi/lo split and the
// swizzled operand-tile stores are the SIMT epilogue, which reads the accumulators with tcgen05.ld.16x256b
// (thread = 2 points x 2 units, all channels).
// Pre-activation jets needed by the reverse sweep are stashed in an L2-resident per-CTA scratch.
// Parameter gradients (weights and biases of every layer) accumulate in TMEM over one tile and are added to
// round-to-nearest fp32 running sums in registers (flush_grads); they are written once, as a per-CTA partial
// vector that reduce_kernel sums in fixed order.
// Round-2 additions, each described where it lives: chunk-0 shadow of the adjoint set + TMEM parking (SmemMap,
// bwd_layer), two W slots with W_2 pinned (w_addr), x^T double buffer, envelope jet ahead of the residual stage
// (envelope_point), loop bound in shared memory, predicated streaming loads.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <type_traits>

#include "pde_launch.h"
#include "pde_tc.h"
#include "pde_tc_core.cuh"

namespace pde {
namespace tc {

constexpr int TP = 64;        // points per tile = UMMA M
constexpr int HP = 64;        // padded hidden width = UMMA N / K
// Epilogue warps: quarter q = w % 4 (16 points), column half h = w / 4 (8 of the 16 columns of a chunk).
constexpr int NEPI = 8;
constexpr int NE = 4;         // elements per thread and chunk: 2 rows x 2 adjacent units
constexpr int NTHREADS = (NEPI + 4) * 32;   // + one warpgroup whose first warp issues the MMAs (rest idle, registers donated)
constexpr int MAXC = 6;       // jet channels the TMEM / smem budget covers
constexpr int COL_R0 = 0;     // TMEM columns: activation / adjoint accumulators (3 interleaved pairs)
constexpr int COL_G = 384;    // gW accumulators: slot s at column COL_G + 64 (s / 2), lane half s % 2
constexpr int COL_SMALL = 448;  // (slot 3) small accumulators, lane half 1: gW0|gb0 at +0, gb_l at +8 l

struct TcArgs {
  int n_h, act, H;
  const float* params;          // fp32: W0t [D][64], b [n_h][64], wL [64], bL
  const unsigned char* wimg;    // per GEMM layer l = 1..n_h-1: hi tile, lo tile (swizzled bf16, rows o, cols i)
  const float* X;
  long long n;
  int num_tiles;
  int prog, n_q, want_grad;
  EnvDev<float> env;
  float alpha, beta_const, energy_const, inv_n;
  const float* f;
  const float* beta;
  const float* energy;
  const float* seed;
  float* partial;               // [grid][PP]
  double* psums;                // [grid][8]
  float4* stash;                // [grid][stash_f4]
  long long PP, stash_f4, off_gW0, off_gb0, off_gW, off_gwL, off_gbL;
  long long* dbg;               // timeline buffer (builds with -DPDE_TC_TIMELINE only), else null
  int dir0;                     // first derivative direction (dimension-split instantiations differentiate along dir0 .. dir0+NDIR-1)
  int mode;                     // 0: envelope + residual program; 1: network jets out (forward only); 2: jet cotangents in
  float* J;                     // mode 1: (n, C) network jets (value, first derivatives) out
  const float* Jbar;            // mode 2: (n, C) cotangents of the network jets in
  // PDE_PROG_FLUX (order-1 instantiations only): face mask and points per face, read by the residual stage together
  // with the point's global index (tile * 64 + tid)
  int faces;
  long long face_n;
};

// ---------------------------------------------------------------- per-element math
// activation derivatives from the two stashed values (sin: (s, c); tanh: (t, 1 - t^2))
__device__ __forceinline__ void act_from_stash(int act, float v0, float v1, float& s0, float& s1, float& s2, float& s3) {
  if (act == 0) {
    s0 = v0; s1 = v1; s2 = -v0; s3 = -v1;
  } else {
    s0 = v0; s1 = v1; s2 = -2.f * v0 * v1; s3 = -2.f * v1 * (1.f - 3.f * v0 * v0);
  }
}
// sin and cos to ~1 ulp for |z| <= 2^15: magic-number rounding of z * 2/pi, three-term Cody-Waite
// reduction by pi/2, minimax polynomials on [-pi/4, pi/4], quadrant fix-up on the sign bits.
// (Callers route larger arguments to the library sincosf.)
__device__ __forceinline__ void sincos_cw(float z, float& s, float& c) {
  const float t = fmaf(z, 0.636619772f, 12582912.f);   // 1.5 * 2^23: the low mantissa bits hold round(z * 2/pi)
  const uint32_t k = __float_as_uint(t);
  const float kf = t - 12582912.f;
  float r = fmaf(kf, -1.57079601e+00f, z);
  r = fmaf(kf, -3.13916473e-07f, r);
  r = fmaf(kf, -5.39030253e-15f, r);
  const float r2 = r * r;
  float sp = fmaf(r2, -1.95152959e-4f, 8.33216087e-3f);
  sp = fmaf(sp, r2, -1.66666546e-1f);
  sp = fmaf(sp * r2, r, r);
  float cp = fmaf(r2, 2.44331571e-5f, -1.38873163e-3f);
  cp = fmaf(cp, r2, 4.16666457e-2f);
  cp = fmaf(cp, r2, -0.5f);
  cp = fmaf(cp, r2, 1.0f);
  const bool odd = (k & 1u) != 0;
  const float a = odd ? cp : sp, b = odd ? sp : cp;
  s = __uint_as_float(__float_as_uint(a) ^ ((k & 2u) << 30));
  c = __uint_as_float(__float_as_uint(b) ^ (((k + 1u) & 2u) << 30));
}
// ---- packed fp32 pairs (Blackwell FFMA2 / FMUL2 / FADD2): one issue slot for two lanes' worth of math
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
  f32x2 d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
  return d;
}
__device__ __forceinline__ void unpk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// sincos_cw on two arguments at once: the reduction and both polynomials in packed arithmetic (14 instead
// of 28 FP instructions), quadrant fix-up per element.  Same operations in the same order as sincos_cw.
__device__ __forceinline__ void sincos_cw2(float z0, float z1, float& s0, float& c0, float& s1, float& c1) {
  const f32x2 z = pk2(z0, z1);
  const f32x2 t = fma2(z, pk2(0.636619772f, 0.636619772f), pk2(12582912.f, 12582912.f));
  const f32x2 kf = add2(t, pk2(-12582912.f, -12582912.f));
  f32x2 r = fma2(kf, pk2(-1.57079601e+00f, -1.57079601e+00f), z);
  r = fma2(kf, pk2(-3.13916473e-07f, -3.13916473e-07f), r);
  r = fma2(kf, pk2(-5.39030253e-15f, -5.39030253e-15f), r);
  const f32x2 r2 = mul2(r, r);
  f32x2 sp = fma2(r2, pk2(-1.95152959e-4f, -1.95152959e-4f), pk2(8.33216087e-3f, 8.33216087e-3f));
  sp = fma2(sp, r2, pk2(-1.66666546e-1f, -1.66666546e-1f));
  sp = fma2(mul2(sp, r2), r, r);
  f32x2 cp = fma2(r2, pk2(2.44331571e-5f, 2.44331571e-5f), pk2(-1.38873163e-3f, -1.38873163e-3f));
  cp = fma2(cp, r2, pk2(4.16666457e-2f, 4.16666457e-2f));
  cp = fma2(cp, r2, pk2(-0.5f, -0.5f));
  cp = fma2(cp, r2, pk2(1.0f, 1.0f));
  float t0, t1, sp0, sp1, cp0, cp1;
  unpk2(t, t0, t1);
  unpk2(sp, sp0, sp1);
  unpk2(cp, cp0, cp1);
  {
    const uint32_t k = __float_as_uint(t0);
    const bool odd = (k & 1u) != 0;
    const float a = odd ? cp0 : sp0, b = odd ? sp0 : cp0;
    s0 = __uint_as_float(__float_as_uint(a) ^ ((k & 2u) << 30));
    c0 = __uint_as_float(__float_as_uint(b) ^ (((k + 1u) & 2u) << 30));
  }
  {
    const uint32_t k = __float_as_uint(t1);
    const bool odd = (k & 1u) != 0;
    const float a = odd ? cp1 : sp1, b = odd ? sp1 : cp1;
    s1 = __uint_as_float(__float_as_uint(a) ^ ((k & 2u) << 30));
    c1 = __uint_as_float(__float_as_uint(b) ^ (((k + 1u) & 2u) << 30));
  }
}
// `big`: warp-uniform flag "some |z| of this chunk is outside the fast range".  One branch for all the
// elements of a thread, so that the independent polynomial chains of the fast path are interleaved.
template <int N>
__device__ __forceinline__ void act_eval(int act, const float (&z)[N], bool big, float (&v0)[N], float (&v1)[N]) {
  if (act == 0) {
    if (big) {
#pragma unroll
      for (int e = 0; e < N; ++e) sincosf(z[e], &v0[e], &v1[e]);
    } else {
      if constexpr (N % 2 == 0) {
#pragma unroll
        for (int e = 0; e < N; e += 2) sincos_cw2(z[e], z[e + 1], v0[e], v1[e], v0[e + 1], v1[e + 1]);
      } else {
#pragma unroll
        for (int e = 0; e < N; ++e) sincos_cw(z[e], v0[e], v1[e]);
      }
    }
  } else {
#pragma unroll
    for (int e = 0; e < N; ++e) {
      v0[e] = tanhf(z[e]);
      v1[e] = 1.f - v0[e] * v0[e];
    }
  }
}

// ---------------------------------------------------------------- envelope + residual program on (value, grad, Lap) jets
// nj: network jets in, cotangents out.  Follows program_point in pde_simt.cuh with the Hessian
// diagonal replaced by its sum.
// The envelope's own jet (B, dB/dx_i, Lap B) depends on the point only: the kernel evaluates it while it waits for the
// first hidden GEMM (envelope_point, into the slots the cotangents take later) and the residual stage reads it back.
template <int D, int ORDER>
__device__ void envelope_point(const TcArgs& a, const float* x, float* out) {
  float b[D], b1[D], b2[D];
#pragma unroll
  for (int i = 0; i < D; ++i) envelope_factor<float>(a.env, i, x[i], b[i], b1[i], b2[i]);
  float B = 1.f;
#pragma unroll
  for (int i = 0; i < D; ++i) B *= b[i];
  float LB = 0.f;
  out[0] = B;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    float e = 1.f;
#pragma unroll
    for (int j = 0; j < D; ++j)
      if (j != i) e *= b[j];
    if constexpr (ORDER >= 1) out[1 + i] = b1[i] * e;
    LB += b2[i] * e;
  }
  if constexpr (ORDER == 2) out[1 + D] = LB;
}
template <int D, int ORDER>
__device__ void program_point_lap(const TcArgs& a, const float* env, const float* cst, float fv, float bt, long long gp,
                                  float (&nj)[1 + (ORDER >= 1 ? D : 0) + (ORDER == 2)], double (&qs)[4], double& gE) {
  constexpr int ND = (ORDER >= 1) ? D : 0;
  const float B = env[0];
  float Bi[D], LB = 0.f;
#pragma unroll
  for (int i = 0; i < D; ++i) Bi[i] = (ORDER >= 1) ? env[1 + i] : 0.f;
  if constexpr (ORDER == 2) LB = env[1 + D];
  const float N0 = nj[0];
  const float u = B * N0;
  float ui[D];
  float lap = 0.f;
#pragma unroll
  for (int i = 0; i < D; ++i) ui[i] = 0.f;
  if constexpr (ORDER >= 1) {
#pragma unroll
    for (int i = 0; i < D; ++i) ui[i] = Bi[i] * N0 + B * nj[1 + i];
  }
  if constexpr (ORDER == 2) {
    lap = LB * N0 + B * nj[1 + ND];
#pragma unroll
    for (int i = 0; i < D; ++i) lap += 2.f * Bi[i] * nj[1 + i];
  }
  const float E = cst[0], w0 = cst[1];   // energy, seed[0] / n (read from global memory once per CTA)
  float ub = 0.f, lapb = 0.f, uib[D];
#pragma unroll
  for (int i = 0; i < D; ++i) uib[i] = 0.f;
  if (a.prog == PDE_PROG_PINN) {
    const float r = a.alpha * lap + (bt - E) * u - fv;
    qs[0] += (double)(r * r);
    const float rb = 2.f * r * w0;
    ub = (bt - E) * rb;
    lapb = a.alpha * rb;
    gE += (double)(-u * rb);
  } else if (a.prog == PDE_PROG_DRM) {
    float g2 = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) g2 += ui[i] * ui[i];
    qs[0] += (double)(a.alpha * g2 - fv * u);
    ub = -fv * w0;
#pragma unroll
    for (int i = 0; i < D; ++i) uib[i] = 2.f * a.alpha * ui[i] * w0;
  } else if (a.prog == PDE_PROG_RAYLEIGH) {
    float g2 = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) g2 += ui[i] * ui[i];
    qs[0] += (double)(a.alpha * g2 + bt * u * u);
    qs[1] += (double)(u * u);
    const float w1 = cst[2];
    ub = 2.f * bt * u * w0 + 2.f * u * w1;
#pragma unroll
    for (int i = 0; i < D; ++i) uib[i] = 2.f * a.alpha * ui[i] * w0;
  } else if (ORDER == 1 && a.prog == PDE_PROG_FLUX) {   // the order-0 / order-2 kernels keep their instruction stream
    int ax, sg;
    flux_face(a.faces, a.face_n, gp, ax, sg);
    const float as = sg > 0 ? a.alpha : -a.alpha;
    float un = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i)
      if (i == ax) un = ui[i];
    const float r = as * un + bt * u - fv;
    qs[0] += (double)(r * r);
    const float rb = 2.f * r * w0;
    ub = bt * rb;
#pragma unroll
    for (int i = 0; i < D; ++i) uib[i] = (i == ax) ? as * rb : 0.f;
  } else {
    const float r = u - fv;
    qs[0] += (double)(r * r);
    ub = 2.f * r * w0;
  }
  float n0b = B * ub;
  if constexpr (ORDER >= 1) {
#pragma unroll
    for (int i = 0; i < D; ++i) {
      n0b += Bi[i] * uib[i];
      float t = B * uib[i];
      if constexpr (ORDER == 2) t += 2.f * Bi[i] * lapb;
      nj[1 + i] = t;
    }
  }
  if constexpr (ORDER == 2) {
    n0b += LB * lapb;
    nj[1 + ND] = B * lapb;
  }
  nj[0] = n0b;
}

// ---------------------------------------------------------------- shared-memory carve-up (bytes from the 1024-aligned base)
template <int D, int C>
struct SmemMap {
  static constexpr int LIMIT = 232448;                    // dynamic shared memory a CTA can opt in to
  static constexpr int set_bytes = 2 * C * TILE_BYTES;
  static constexpr int par_floats = D * 64 + 4 * 64 + 64 + 4;
  static constexpr int red_floats = (2 * 64 * C > 256) ? 2 * 64 * C : 256;   // also [4][64] at the end
  // everything but the operand sets, W and the chunk-0 shadow
  static constexpr int rest = 4096 + 1024 * (D > 0 ? D : 1) + par_floats * 4 + 64 * D * 4 + 64 * C * 4 + red_floats * 4 + 128;
  // Chunk-0 shadow of the adjoint set (reverse sweep): columns 0..15 of the 2 C adjoint tiles in an unswizzled K-major
  // layout (2 KB per tile), so that a reverse layer can publish its first chunk while the previous layer's wgrad still
  // reads the adjoint set proper.  Where it only fits with two W slots, W_1 stays and W_2 / W_3 share the second slot.
  static constexpr int shadow_if = 2 * C * 2048;
  static constexpr bool fits3 = 2 * set_bytes + 3 * 2 * TILE_BYTES + shadow_if + rest <= LIMIT;
  static constexpr bool fits2 = 2 * set_bytes + 2 * 2 * TILE_BYTES + shadow_if + rest <= LIMIT;
  static constexpr bool shadow = (C <= 5) && (fits3 || fits2);
  static constexpr int w_slots = (C <= 5) ? ((shadow && !fits3) ? 2 : 3) : 1;   // 3: every hidden W resident
  static constexpr int off_T1 = 0;                        // activations A_l (operand of fwd / wgrad)
  static constexpr int off_T2 = off_T1 + set_bytes;       // adjoints Zb_l (operand of dgrad / wgrad)
  static constexpr int off_W = off_T2 + set_bytes;        // W_l hi, lo per slot
  static constexpr int w_bytes = w_slots * 2 * TILE_BYTES;
  static constexpr int off_Z0 = off_W + w_bytes;          // chunk-0 shadow of the adjoint set
  static constexpr int off_XT = off_Z0 + (shadow ? shadow_if : 0);   // x^T hi, lo (8 rows x 128 B each), rows j<D: x_j, row D: ones; two buffers (tile parity)
  static constexpr int off_E = off_XT + 4096;             // indicator tiles E_0..E_{D-1}: row n all ones
  static constexpr int off_par = off_E + 1024 * (D > 0 ? D : 1);   // fp32 W0t [D][64], b [4][64], wL [64], bL(+pad)
  static constexpr int off_X = off_par + par_floats * 4;  // X tile [64][D]
  static constexpr int off_nb = off_X + 64 * D * 4;       // cotangents of the network jets [64][C]
  static constexpr int off_red = off_nb + 64 * C * 4;     // output-layer partial sums [2][64][C]
  static constexpr int off_bar = off_red + red_floats * 4;
  static constexpr int total = off_bar + 128;
  static_assert(total <= LIMIT, "shared-memory plan does not fit");
};

// explicit state-space accesses (pointers reached through the argument struct are generic otherwise)
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void stsm_x4(uint32_t addr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.shared.b16 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
// The stash is rewritten every tile and dead after the tile's reverse sweep, but an L2 line that is merely dirty is
// still written back to HBM when it is evicted.  Stash traffic carries an L2 evict_last policy and the streamed
// inputs (X, f, beta) evict_first, so that the one-pass inputs do not push stash lines out.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void stash_store(float4* p, float4 v, uint64_t pol) {
  asm volatile("st.global.cg.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ float4 stash_load(const float4* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.cg.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
  return v;
}
// one-pass inputs
__device__ __forceinline__ float stream_load(const float* p, uint64_t pol) {
  float v;
  asm volatile("ld.global.cg.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
  return v;
}
// the same under a predicate (0 when it is false).  One asm block, so that the register is written by the predicated
// load itself: a select after the load would make the warp wait for the DRAM round trip right where it was issued.
__device__ __forceinline__ float stream_load_if(const float* p, uint64_t pol, bool pred) {
  float v;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %3, 0;\n\t"
      "mov.f32 %0, 0f00000000;\n\t"
      "@p ld.global.cg.L2::cache_hint.f32 %0, [%1], %2;\n\t"
      "}"
      : "=f"(v)
      : "l"(p), "l"(pol), "r"((int)pred));
  return v;
}
// stashed vector <-> the thread's element array
__device__ __forceinline__ void to_arr(const float4& sv, float (&v)[4]) { v[0] = sv.x; v[1] = sv.y; v[2] = sv.z; v[3] = sv.w; }
__device__ __forceinline__ float4 from_arr(const float (&v)[4]) { return make_float4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ void named_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// UMMA descriptors as "constant high word + 14-bit start address (16-byte units) in the low word":
// K-major / MN-major Tile64 views (LBO 16 / 8192 bytes, SBO 1024 bytes, version 1, SWIZZLE_128B)
constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO | version | layout type
constexpr uint32_t DESC_HI_G2 = (2048u >> 4) | (1u << 14) | (2u << 29);   // MN-major view of a paired channel: 8-row groups 2 KB apart
constexpr uint32_t DESC_K_LBO = (16u >> 4) << 16;      // low word, next to the start address
constexpr uint32_t DESC_MN_LBO = (8192u >> 4) << 16;
// Channel pairs stacked along M.  A tcgen05.mma whose operands both come from shared memory costs what its A
// tile costs to read, and an M = 128 instruction (52 cycles) is cheaper than two M = 64 ones (2 x 39): channels 2p and 2p+1
// of an operand set share a pair of 16 KB blocks (hi, lo) with their 8-row groups interleaved (channel c & 1 of point
// group g at row group 2g + (c & 1)), so that one M = 128 K-major descriptor covers both in the forward and dgrad GEMMs;
// the accumulator rows land in TMEM exactly where the two M = 64 accumulators used to be interleaved by hand, only with
// the roles of (lane half, row half) swapped (pick_ch).  An odd last channel keeps the plain (hi tile, lo tile) layout.
// In the MN-major views (wgrad, first layer, biases) a paired channel simply has its row groups 2 KB apart.
__host__ __device__ constexpr bool ch_paired(int c, int C) { return (c | 1) < C; }
__host__ __device__ constexpr uint32_t ch_base(int c, int C) {   // bytes from the set's start to channel c's first row group (hi part)
  return ch_paired(c, C) ? (uint32_t)(c >> 1) * 4u * TILE_BYTES + (uint32_t)(c & 1) * 1024u : (uint32_t)c * 2u * TILE_BYTES;
}
__host__ __device__ constexpr uint32_t ch_lo(int c, int C) { return ch_paired(c, C) ? 2u * TILE_BYTES : (uint32_t)TILE_BYTES; }   // hi -> lo part
__host__ __device__ constexpr uint32_t ch_kstep_mn(int c, int C) { return ch_paired(c, C) ? 4096u : 2048u; }   // 16 points in the MN-major view
__host__ __device__ constexpr uint32_t ch_hi_mn(int c, int C) { return ch_paired(c, C) ? DESC_HI_G2 : DESC_HI; }
// the same for the chunk-0 shadow (2 KB per channel part, row groups 256 bytes)
__host__ __device__ constexpr uint32_t z0_base_of(int c, int C) { return ch_paired(c, C) ? (uint32_t)(c >> 1) * 8192u + (uint32_t)(c & 1) * 256u : (uint32_t)c * 4096u; }
__host__ __device__ constexpr uint32_t z0_lo(int c, int C) { return ch_paired(c, C) ? 4096u : 2048u; }
// one tcgen05.mma from 32-bit descriptor words
__device__ __forceinline__ void mma_k(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                      uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(d_tmem),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- the kernel
// Warps 0..7: epilogue (quarter q = w % 4 owns points 16q..16q+15, half h = w / 4 owns 8 of the 16
// columns of a chunk).  Warp 8: one elected thread issues every tcgen05.mma.
// Hand-offs (all mbarriers, one phase bit each, flipped once per use):
//   bar_chunk[j]  8 arrivals   epilogue -> issuer : operand columns 16j..16j+15 (= K step j) are in smem
//   bar_d         commit       issuer -> epilogue : the accumulators the next step reads are complete
//   bar_w         commit       issuer -> epilogue : every MMA that reads the operand sets has completed
// Accumulator regions ping-pong (R0/R1) so that the MMAs of step s+1 run while step s is still
// being read; a step's K-step-j MMAs are issued as soon as chunk j has been written.
// NDIR < D: dimension-split instantiation — jets along the NDIR directions dir0 .. dir0+NDIR-1 only (value, NDIR first
// derivatives, the partial Laplacian over those directions); jet modes only.  The 5-D PINN step, whose 7 channels do
// not fit on chip, is two such passes (3 + 2 directions) around a pointwise residual kernel (tc_pinn_split).
template <int D, int ORDER, int ACT, int NDIR = D>
__global__ void __launch_bounds__(NTHREADS, 1) tc_kernel(const TcArgs a) {
  constexpr int ND = (ORDER >= 1) ? NDIR : 0;
  constexpr bool SPLIT = (NDIR != D);
  const int dir0 = SPLIT ? a.dir0 : 0;
  constexpr int LAP = (ORDER == 2) ? 1 : 0;
  constexpr int C = 1 + ND + LAP;
  constexpr int NV = 2 + ND + LAP;  // stashed values per (point, unit, layer)
  static_assert(C <= MAXC, "too many jet channels for the TMEM / smem budget");
  using SM = SmemMap<D, C>;
  constexpr int WS = SM::w_slots;
  constexpr bool WRES = (WS == 3);
  constexpr bool SHADOW = SM::shadow;

  extern __shared__ __align__(1024) unsigned char sm[];
  float* sPar = reinterpret_cast<float*>(sm + SM::off_par);
  float* sW0t = sPar;                 // [D][64]
  float* sB = sPar + D * 64;          // [4][64]
  float* sWL = sB + 4 * 64;           // [64], then bL
  float* sX = reinterpret_cast<float*>(sm + SM::off_X);
  float* sNb = reinterpret_cast<float*>(sm + SM::off_nb);
  float* sRed = reinterpret_cast<float*>(sm + SM::off_red);
  uint64_t* bar_chunk = reinterpret_cast<uint64_t*>(sm + SM::off_bar);   // [4]
  uint64_t* bar_d = bar_chunk + 4;
  uint64_t* bar_w = bar_chunk + 5;
  uint64_t* bar_own = bar_chunk + 6;   // issuer-private: "everything I issued so far has completed"
  uint64_t* bar_wt = bar_chunk + 7;    // bulk copy of a W tile pair has landed (non-resident W only)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_chunk + 8);
  int* sTileEnd = reinterpret_cast<int*>(bar_chunk + 14);   // the epilogue's loop bound (see there)
  // (bar_chunk + 9 is unused)
  float* sMx = reinterpret_cast<float*>(bar_chunk + 10);   // per-tile maximum cotangent of warps 0 and 1

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_h = a.n_h;
  constexpr int act = ACT;
  const bool do_bwd = a.want_grad != 0;
  const uint32_t sbase = smem_u32(sm);
  const uint32_t sT1 = sbase + SM::off_T1, sT2 = sbase + SM::off_T2, sWT = sbase + SM::off_W;
  const uint32_t sXT = sbase + SM::off_XT, sET = sbase + SM::off_E, sZ0 = sbase + SM::off_Z0;

  // W slots: 3 = layer l in slot l-1; 1 = one slot for all, refilled before every GEMM layer; 2 = W_2 stays in slot 0,
  // W_1 and W_3 take turns in slot 1: each is fetched a whole layer before it is needed (W_3 once the forward GEMM of
  // layer 1 has completed, W_1 once dgrad_3 has), so that copy is never waited for.
  auto w_addr = [&](int l) { return sWT + (WS == 3 ? l - 1 : (WS == 2 ? (l == 2 ? 0 : 1) : 0)) * 2 * TILE_BYTES; };
  // ---- one-time setup (all warps)
  for (int i = tid; i < D * 64 + n_h * 64; i += NTHREADS) sPar[i] = a.params[i];
  for (int i = tid; i < 64 + 1; i += NTHREADS) sWL[i] = a.params[D * 64 + n_h * 64 + i];
  if (tid == 0 && a.mode == 0) {
    // loop-invariant scalars of the residual stage
    sWL[65] = a.energy ? a.energy[0] : a.energy_const;
    sWL[66] = (a.seed ? a.seed[0] : 1.f) * a.inv_n;
    sWL[67] = (a.seed && a.prog == PDE_PROG_RAYLEIGH ? a.seed[1] : 1.f) * a.inv_n;
  }
  for (int i = tid; i < (1024 * (D > 0 ? D : 1)) / 4; i += NTHREADS) {
    const int n = i / 256, w = i % 256;  // tile n, 32-bit word w: row = w / 32
    reinterpret_cast<uint32_t*>(sm + SM::off_E)[i] = ((w >> 5) == n) ? ONE_X2 : 0u;
  }
  for (int i = tid; i < 1024; i += NTHREADS) {
    const int t = (i / 256) & 1, w = i % 256;   // hi, lo tile of either buffer
    reinterpret_cast<uint32_t*>(sm + SM::off_XT)[i] = (t == 0 && (w >> 5) == D) ? ONE_X2 : 0u;
  }
  {
    // resident: every hidden layer's W; otherwise W_1 (later layers are streamed by the issuer)
    const uint4* src = reinterpret_cast<const uint4*>(a.wimg);
    uint4* dst = reinterpret_cast<uint4*>(sm + SM::off_W);
    for (int l = 1; l <= (n_h - 1 < WS ? n_h - 1 : WS); ++l) {
      dst = reinterpret_cast<uint4*>(sm + SM::off_W + (w_addr(l) - sWT));
      for (int i = tid; i < 2 * TILE_BYTES / 16; i += NTHREADS) dst[i] = src[(l - 1) * (2 * TILE_BYTES / 16) + i];
    }
  }
  if (tid == 0) {
    for (int j = 0; j < 4; ++j) mbar_init(&bar_chunk[j], NEPI);
    mbar_init(bar_d, 1);
    mbar_init(bar_w, 1);
    mbar_init(bar_own, 1);
    mbar_init(bar_wt, 1);
    fence_mbar_init();
    if (sbase & 1023u) __trap();   // SWIZZLE_128B tiles need the 1024-byte alignment the declaration asks for
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // this CTA's contiguous range of tiles
  const int tile_begin = (int)(((long long)a.num_tiles * blockIdx.x) / gridDim.x);
  const int tile_end = (int)(((long long)a.num_tiles * (blockIdx.x + 1)) / gridDim.x);

#ifdef PDE_TC_TIMELINE
  // development timeline: (event id, clock) pairs of CTA 0, epilogue warp 0 and the issuer
  int dbg_n = 0;
  auto TS = [&](int id) {
    if (a.dbg && blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == NEPI) && dbg_n < 2000) {
      long long* p = a.dbg + (warp == 0 ? 0 : 4096) + 2 * dbg_n;
      p[0] = id; p[1] = clock64();
      ++dbg_n;
    }
  };
  // every epilogue warp: arrival at the CTA-wide barriers (id, clock), 500 events per warp
  int dbgw_n = 0;
  auto TSW = [&](int id) {
    if (a.dbg && blockIdx.x == 0 && lane == 0 && warp < NEPI && dbgw_n < 500) {
      long long* p = a.dbg + 8192 + warp * 1024 + 2 * dbgw_n;
      p[0] = id; p[1] = clock64();
      ++dbgw_n;
    }
  };
#else
  auto TS = [](int) {};
  auto TSW = [](int) {};
#endif
  // accumulator address of jet channel c in region r: pair c/2 at columns 64 (c/2), lane half c%2
  auto d_addr = [&](int r, int c) { return taddr_of(tmem, 16 * (c & 1), COL_R0 + 192 * r + 64 * (c >> 1)); };

  if (warp >= NEPI) {
    // =====================================================================================
    // MMA issuer (warp NEPI); its warpgroup hands its registers to the epilogue.  The warp runs
    // the loops convergently and one elected lane issues, so descriptor arithmetic stays uniform.
    // =====================================================================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");   // 256 x 208 + 128 x 88 = the 384 x 168 registers the CTA launches with
    if (warp == NEPI) {
      constexpr uint32_t ID_FWD = make_idesc(64, 64, 0, 0);   // A K-major, B K-major
      constexpr uint32_t ID_FWD2 = make_idesc(128, 64, 0, 0), ID_DG2 = make_idesc(128, 64, 0, 1);   // channel pairs
      constexpr uint32_t ID_DG = make_idesc(64, 64, 0, 1);    // A K-major, B MN-major (W viewed as W^T)
      constexpr uint32_t ID_WG = make_idesc(64, 64, 1, 1);    // A, B MN-major (contraction over points)
      constexpr uint32_t ID_SM = make_idesc(64, 8, 1, 0);     // A MN-major, B K-major, N = 8
      constexpr uint32_t TD = TILE_BYTES >> 4;                // one tile in descriptor address units
      const uint32_t tm = __shfl_sync(0xffffffffu, tmem, 0);
      // low descriptor words (start address in 16-byte units | LBO) of the K-major / MN-major views
      const uint32_t kT1K = (sT1 >> 4) | DESC_K_LBO, kT1M = (sT1 >> 4) | DESC_MN_LBO;
      const uint32_t kT2K = (sT2 >> 4) | DESC_K_LBO, kT2M = (sT2 >> 4) | DESC_MN_LBO;
      const uint32_t kXT0 = (sXT >> 4) | DESC_K_LBO, kETK = (sET >> 4) | DESC_K_LBO;
      uint32_t ph_chunk = 0, ph_own = 0, ph_wt = 0;
      int reg = 0;   // region the next D-producing GEMM writes
      int cur_w = 1;   // layer whose W sits in the shared slot (non-resident W)
      // chunk-0 shadow (unswizzled K-major: LBO 128 = next core matrix along K, SBO 256 = next 8 rows)
      const uint32_t kZ0 = (sZ0 >> 4) | ((128u >> 4) << 16);
      constexpr uint32_t DESC_HI_Z0 = (256u >> 4) | (1u << 14);
      // Non-resident W (6 channels): one tile-pair buffer, refilled with a bulk copy.  need_w(l) makes W_l current:
      // drain my MMAs (they may read the buffer), copy, wait.  In the reverse sweep the copy of W_{l-1} is started as
      // soon as dgrad_l has completed — wgrad_l, which runs for another ~2.6 k cycles, does not read W — so only its
      // arrival is waited for when layer l-1 starts.
      bool w_loading = false;
      auto start_w_load = [&](int l) {
        if (elect_one()) {
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar_wt)), "r"(2 * TILE_BYTES) : "memory");
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(w_addr(l)),
                       "l"(a.wimg + (size_t)(l - 1) * 2 * TILE_BYTES), "r"(2 * TILE_BYTES), "r"(smem_u32(bar_wt))
                       : "memory");
        }
        __syncwarp();
        cur_w = l;
        w_loading = true;
      };
      auto need_w = [&](int l) {
        if (WRES) return;
        if (WS == 2 && l == 2) return;
        // (two slots: the copy was normally started a layer ago, see below, and only its arrival is waited for;
        //  forward-only launches find W_3 in the slot when the next tile asks for W_1 and take the slow way)
        if (cur_w != l) {
          if (elect_one()) mma_commit(bar_own);
          __syncwarp();
          mbar_wait(bar_own, ph_own);
          ph_own ^= 1;
          start_w_load(l);
        }
        if (w_loading) {
          mbar_wait(bar_wt, ph_wt);
          ph_wt ^= 1;
          w_loading = false;
        }
      };
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        // ---- forward GEMMs of layers 1..n_h-1, K step j as soon as chunk j of A_{l-1} is there
        for (int l = 1; l < n_h; ++l) {
          // fresh copies of the descriptor bases: without them ptxas precomputes every (base + tile offset) of the unrolled
          // issue loops outside the tile loop, ~40 values for the small-C variants, and reloads them from local memory
          // in front of every K step (the 5- and 6-channel variants keep them in registers and are faster left alone)
          uint32_t kT1K_ = kT1K, kT1M_ = kT1M, kT2K_ = kT2K, kT2M_ = kT2M, kXT0_ = kXT0, kETK_ = kETK, kZ0_ = kZ0;
          if constexpr (C <= 4) asm volatile("" : "+r"(kT1K_), "+r"(kT1M_), "+r"(kT2K_), "+r"(kT2M_), "+r"(kXT0_), "+r"(kETK_), "+r"(kZ0_));
          const uint32_t kW = (w_addr(l) >> 4) | DESC_K_LBO;
          const uint32_t dbase = tm + COL_R0 + 192 * reg;
          need_w(l);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            mbar_wait(&bar_chunk[j], ph_chunk);
            tc_fence_after();
            TS(100 + 10 * l + j);
            // the epilogue has consumed the accumulators of layer 1, so nothing reads W_1 any more
            if (WS == 2 && j == 0 && l == 2 && n_h - 1 == 3) start_w_load(3);
            if (elect_one()) {
#pragma unroll
              for (int c = 0; c < C; ++c) {
                if (ch_paired(c, C) && (c & 1)) continue;   // covered by its partner's M = 128 instructions
                const uint32_t d = dbase + 64 * (c >> 1);
                const uint32_t ah = kT1K_ + (ch_base(c, C) >> 4) + 2 * j, al = ah + (ch_lo(c, C) >> 4);
                const uint32_t id = ch_paired(c, C) ? ID_FWD2 : ID_FWD;
                mma_k(d, ah, DESC_HI, kW + 2 * j, DESC_HI, id, j > 0 ? 1u : 0u);
                mma_k(d, al, DESC_HI, kW + 2 * j, DESC_HI, id, 1u);
                mma_k(d, ah, DESC_HI, kW + TD + 2 * j, DESC_HI, id, 1u);
              }
            }
            __syncwarp();
          }
          if (elect_one()) mma_commit(bar_d);
          __syncwarp();
          ph_chunk ^= 1;
          reg ^= 1;
        }
        if (!do_bwd) continue;
        // ---- reverse sweep
        for (int l = n_h - 1; l >= 1; --l) {
          // fresh copies of the descriptor bases: without them ptxas precomputes every (base + tile offset) of the unrolled
          // issue loops outside the tile loop, ~40 values for the small-C variants, and reloads them from local memory
          // in front of every K step (the 5- and 6-channel variants keep them in registers and are faster left alone)
          uint32_t kT1K_ = kT1K, kT1M_ = kT1M, kT2K_ = kT2K, kT2M_ = kT2M, kXT0_ = kXT0, kETK_ = kETK, kZ0_ = kZ0;
          if constexpr (C <= 4) asm volatile("" : "+r"(kT1K_), "+r"(kT1M_), "+r"(kT2K_), "+r"(kT2M_), "+r"(kXT0_), "+r"(kETK_), "+r"(kZ0_));
          const uint32_t kW = (w_addr(l) >> 4) | DESC_MN_LBO;
          const uint32_t dbase = tm + COL_R0 + 192 * reg;
          need_w(l);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            mbar_wait(&bar_chunk[j], ph_chunk);
            tc_fence_after();
            TS(200 + 10 * l + j);
            if (WS == 2 && j == 0 && l == 2 && n_h - 1 == 3) start_w_load(1);   // dgrad_3 has been consumed
            // dgrad: Ab_{l-1,c} += Zb_{l,c}[:, K step j] W_l[K step j, :]
            if (SHADOW && j == 0 && l < n_h - 1) {
              // below the top layer the first chunk of the adjoints sits in the shadow
              if (elect_one()) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                  if (ch_paired(c, C) && (c & 1)) continue;
                  const uint32_t d = dbase + 64 * (c >> 1);
                  const uint32_t zh = kZ0_ + (z0_base_of(c, C) >> 4), zl = zh + (z0_lo(c, C) >> 4);
                  const uint32_t id = ch_paired(c, C) ? ID_DG2 : ID_DG;
                  mma_k(d, zh, DESC_HI_Z0, kW, DESC_HI, id, 0u);
                  mma_k(d, zl, DESC_HI_Z0, kW, DESC_HI, id, 1u);
                  mma_k(d, zh, DESC_HI_Z0, kW + TD, DESC_HI, id, 1u);
                }
              }
            } else if (elect_one()) {
#pragma unroll
              for (int c = 0; c < C; ++c) {
                if (ch_paired(c, C) && (c & 1)) continue;
                const uint32_t d = dbase + 64 * (c >> 1);
                const uint32_t zh = kT2K_ + (ch_base(c, C) >> 4) + 2 * j, zl = zh + (ch_lo(c, C) >> 4);
                const uint32_t id = ch_paired(c, C) ? ID_DG2 : ID_DG;
                mma_k(d, zh, DESC_HI, kW + 128 * j, DESC_HI, id, j > 0 ? 1u : 0u);
                mma_k(d, zl, DESC_HI, kW + 128 * j, DESC_HI, id, 1u);
                mma_k(d, zh, DESC_HI, kW + TD + 128 * j, DESC_HI, id, 1u);
              }
            }
            __syncwarp();
          }
          const bool refill_next = (WS == 1) && l > 1;
          if (elect_one()) {
            mma_commit(bar_d);
            if (refill_next) mma_commit(bar_own);   // "dgrad_l has completed": the W buffer may be refilled
          }
          __syncwarp();
          ph_chunk ^= 1;
          reg ^= 1;
          // wgrad: gW_l(tile) = sum_c Zb_{l,c}^T A_{l-1,c}   (K = 64 points);  bias: gb_l(tile) = Zb_{l,0}^T 1.
          // The accumulators start from zero every tile (the epilogue adds them to the running fp32
          // sums, see flush_grads) and the small cross terms go first: the tensor core truncates
          // when it accumulates, so the error of an update scales with the accumulator's magnitude.
          if (elect_one()) {
            const int sl = l - 1;
            const uint32_t d = tm + ((16 * (sl & 1)) << 16) + COL_G + 64 * (sl >> 1);
#pragma unroll
            for (int c = 0; c < C; ++c) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                const uint32_t zh = kT2M_ + ((ch_base(c, C) + ks * ch_kstep_mn(c, C)) >> 4), zl = zh + (ch_lo(c, C) >> 4);
                const uint32_t ah = kT1M_ + ((ch_base(c, C) + ks * ch_kstep_mn(c, C)) >> 4), al = ah + (ch_lo(c, C) >> 4);
                mma_k(d, zl, ch_hi_mn(c, C), ah, ch_hi_mn(c, C), ID_WG, (c == 0 && ks == 0) ? 0u : 1u);
                mma_k(d, zh, ch_hi_mn(c, C), al, ch_hi_mn(c, C), ID_WG, 1u);
              }
            }
#pragma unroll
            for (int c = 0; c < C; ++c) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                mma_k(d, kT2M_ + ((ch_base(c, C) + ks * ch_kstep_mn(c, C)) >> 4), ch_hi_mn(c, C),
                      kT1M_ + ((ch_base(c, C) + ks * ch_kstep_mn(c, C)) >> 4), ch_hi_mn(c, C), ID_WG, 1u);
            }
            const uint32_t db = tm + (16u << 16) + COL_SMALL + 8 * l;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              mma_k(db, kT2M_ + ((ch_lo(0, C) + ks * ch_kstep_mn(0, C)) >> 4), ch_hi_mn(0, C), kETK_ + 2 * ks, DESC_HI, ID_SM, ks == 0 ? 0u : 1u);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) mma_k(db, kT2M_ + ((ks * ch_kstep_mn(0, C)) >> 4), ch_hi_mn(0, C), kETK_ + 2 * ks, DESC_HI, ID_SM, 1u);
            mma_commit(bar_w);
          }
          __syncwarp();
          if (refill_next) {
            mbar_wait(bar_own, ph_own);
            ph_own ^= 1;
            start_w_load(l - 1);   // under wgrad_l
          }
        }
        // ---- first layer: [gW0 | gb0] += Zb_{0,0}^T [x | 1] + sum_i Zb_{0,i}^T e_i
        {
          // fresh copies of the descriptor bases: without them ptxas precomputes every (base + tile offset) of the unrolled
          // issue loops outside the tile loop, ~40 values for the small-C variants, and reloads them from local memory
          // in front of every K step (the 5- and 6-channel variants keep them in registers and are faster left alone)
          uint32_t kT1K_ = kT1K, kT1M_ = kT1M, kT2K_ = kT2K, kT2M_ = kT2M, kXT0_ = kXT0, kETK_ = kETK, kZ0_ = kZ0;
          if constexpr (C <= 4) asm volatile("" : "+r"(kT1K_), "+r"(kT1M_), "+r"(kT2K_), "+r"(kT2M_), "+r"(kXT0_), "+r"(kETK_), "+r"(kZ0_));
#pragma unroll
          for (int j = 0; j < 4; ++j) mbar_wait(&bar_chunk[j], ph_chunk);
          tc_fence_after();
          ph_chunk ^= 1;
          if (elect_one()) {
            const uint32_t d = tm + (16u << 16) + COL_SMALL;
            const uint32_t kXTK = kXT0_ + ((tile & 1) << 7);   // this tile's x^T buffer (2048 B apart)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              mma_k(d, kT2M_ + ((ch_lo(0, C) + ks * ch_kstep_mn(0, C)) >> 4), ch_hi_mn(0, C), kXTK + 2 * ks, DESC_HI, ID_SM, ks == 0 ? 0u : 1u);
              mma_k(d, kT2M_ + ((ks * ch_kstep_mn(0, C)) >> 4), ch_hi_mn(0, C), kXTK + 64 + 2 * ks, DESC_HI, ID_SM, 1u);
            }
#pragma unroll
            for (int i = 0; i < ND; ++i) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                mma_k(d, kT2M_ + ((ch_base(1 + i, C) + ch_lo(1 + i, C) + ks * ch_kstep_mn(1 + i, C)) >> 4), ch_hi_mn(1 + i, C),
                      kETK_ + 64 * (dir0 + i) + 2 * ks, DESC_HI, ID_SM, 1u);
            }
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) mma_k(d, kT2M_ + ((ks * ch_kstep_mn(0, C)) >> 4), ch_hi_mn(0, C), kXTK + 2 * ks, DESC_HI, ID_SM, 1u);
#pragma unroll
            for (int i = 0; i < ND; ++i) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                mma_k(d, kT2M_ + ((ch_base(1 + i, C) + ks * ch_kstep_mn(1 + i, C)) >> 4), ch_hi_mn(1 + i, C),
                      kETK_ + 64 * (dir0 + i) + 2 * ks, DESC_HI, ID_SM, 1u);   // E tile of direction dir0 + i: column dir0 + i of gW0
            }
            mma_commit(bar_w);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // =====================================================================================
    // epilogue warps
    // =====================================================================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 208;");
    const int q = warp & 3, h = (warp >> 2) & 1;
    int rows[2];                                        // this thread's points (tile rows)
    rows[0] = 16 * q + (lane >> 2);
    rows[1] = rows[0] + 8;
    const int cq = 2 * (lane & 3);                      // column offset inside an 8-column block
    // stmatrix row address of this thread: matrix i = lane/8 = (hi r0-rows, hi r1-rows, lo r0-rows, lo r1-rows)
    const int sm_row = 16 * q + 8 * ((lane >> 3) & 1) + (lane & 7);
    const int sm_tile = lane >> 4;
    const uint32_t sm_base = (uint32_t)(sm_tile * TILE_BYTES) + ((sm_row >> 3) << 10) + ((sm_row & 7) << 7);
    const int sm_r7 = sm_row & 7;
    float* part = a.partial + (long long)blockIdx.x * a.PP;
    float4* stash = a.stash + (long long)blockIdx.x * a.stash_f4 + warp * (NV * 32) + lane;
    // this thread's part of a 16x256b accumulator fragment (rows lane/4 and lane/4 + 8, two columns each);
    // only valid after tcgen05.wait::ld
    auto pick = [&](const float (&t)[4], float (&v)[NE]) {
#pragma unroll
      for (int e = 0; e < 4; ++e) v[e] = t[e];
    };
    // accumulator fragments of channel c from the raw 16x256b loads (one per channel slot, as issued): a paired channel's
    // two rows come from the two loads of its pair (lane halves = row halves), its columns from word pair c & 1
    auto pick_ch = [&](const float (&t)[C][4], const int c, float (&v)[NE]) {
      if (ch_paired(c, C)) {
        const int p = c & ~1, k = 2 * (c & 1);
        v[0] = t[p][k]; v[1] = t[p][k + 1]; v[2] = t[p + 1][k]; v[3] = t[p + 1][k + 1];
      } else {
        pick(t[c], v);
      }
    };
    // (zeroed, then set: initialising them in the declaration swaps two issuer registers of the 5- and 6-channel variants)
    uint64_t pol_stash = 0, pol_stream = 0;
    pol_stash = l2_policy_evict_last();
    pol_stream = l2_policy_evict_first();
    uint32_t ph_d = 0, ph_w = 0;
    int reg = 0;   // region the next D-consuming step reads
    bool w_pending = false;   // a bar_w commit has been issued that nobody waited for yet

    double qs[4] = {0.0, 0.0, 0.0, 0.0};
    double gE = 0.0;
    // Six-channel variants are over the register budget and ptxas would keep these running sums (used once per tile, by
    // the residual stage of warps 0 and 1) in local memory, whose reloads miss L1 behind the stash traffic.  They are kept
    // in the last free TMEM columns instead (lane half 1 of the small accumulators' slot, columns 32..47).
    constexpr bool PARK_Q = (C == 6);
    const uint32_t qpark = taddr_of(tmem, 32 * q + 16, COL_SMALL + 32);
    auto q_load = [&](double (&t)[4], double& g) {
      uint32_t w0[4], w1[4];
      tmem_ld_16x256b_u32(qpark, w0);
      tmem_ld_16x256b_u32(qpark + 8, w1);
      tmem_ld_wait();
      t[0] = __hiloint2double((int)w0[1], (int)w0[0]);
      t[1] = __hiloint2double((int)w0[3], (int)w0[2]);
      t[2] = t[3] = 0.0;
      g = __hiloint2double((int)w1[1], (int)w1[0]);
    };
    auto q_store = [&](const double (&t)[4], const double g) {
      const uint32_t w0[4] = {(uint32_t)__double2loint(t[0]), (uint32_t)__double2hiint(t[0]), (uint32_t)__double2loint(t[1]), (uint32_t)__double2hiint(t[1])};
      const uint32_t w1[4] = {(uint32_t)__double2loint(g), (uint32_t)__double2hiint(g), 0u, 0u};
      tmem_st_16x256b_u32(qpark, w0);
      tmem_st_16x256b_u32(qpark + 8, w1);
      tmem_st_wait();
    };
    if constexpr (PARK_Q) {
      if (tid < TP) q_store(qs, gE);
    }
    float gwl[4][2];   // output-layer weight gradient partials of this thread's columns
#pragma unroll
    for (int j = 0; j < 4; ++j) gwl[j][0] = gwl[j][1] = 0.f;
    float gbl = 0.f;   // output bias gradient partial (program threads)
    float adj_scale = 0.f;   // power-of-two scale the running gradient sums carry (0 = not chosen yet)
    float cur_scale = 1.f;   // scale of the current tile's adjoints

    // write 4 values (2 rows x 2 adjacent units) of every channel of chunk j into an operand set
    auto pack_chunk = [&](const float (&v)[C][NE], uint32_t (&pk)[C][NE]) {
#pragma unroll
      for (int c = 0; c < C; ++c) {
        split2(v[c][0], v[c][1], pk[c][0], pk[c][2]);
        split2(v[c][2], v[c][3], pk[c][1], pk[c][3]);
      }
    };
    // paired channels: the lo part is a pair block (two tiles) further, the 8-row groups are 2 KB apart
    const uint32_t pair_extra = (uint32_t)(sm_tile * TILE_BYTES) + ((sm_row >> 3) << 10);
    auto put_chunk = [&](uint32_t set, int j, const uint32_t (&pk)[C][NE]) {
      const uint32_t addr = set + sm_base + ((((2 * j + h) ^ sm_r7) & 7) << 4);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const uint32_t ac = addr + ch_base(c, C) + (ch_paired(c, C) ? pair_extra : 0u);
        stsm_x4(ac, pk[c][0], pk[c][1], pk[c][2], pk[c][3]);
      }
    };
    // chunk 0 of the adjoints into the shadow (unswizzled: 8-row group g at 256 g, K half h at +128, row at +16 (row & 7))
    const uint32_t z0_base = sZ0 + (uint32_t)(sm_tile * 2048) + ((sm_row >> 3) << 8) + (h << 7) + ((sm_row & 7) << 4);
    auto put_shadow = [&](const uint32_t (&pk)[C][NE]) {
#pragma unroll
      for (int c = 0; c < C; ++c)
        stsm_x4(z0_base + z0_base_of(c, C) + (ch_paired(c, C) ? (pair_extra >> 2) : 0u), pk[c][0], pk[c][1], pk[c][2], pk[c][3]);
    };
    // ... and from there into the adjoint set proper: every warp moves the 16 rows x 16 bytes per tile it wrote itself
    auto copy_shadow = [&]() {
      const int t = lane >> 4, row = 16 * q + (lane & 15);
      const uint32_t src = sZ0 + (uint32_t)(t * 2048) + ((row >> 3) << 8) + (h << 7) + ((row & 7) << 4);
      const uint32_t dst = sT2 + (uint32_t)(t * TILE_BYTES) + tile_off(row, h);
      const uint32_t dextra = (uint32_t)(t * TILE_BYTES) + ((row >> 3) << 10);   // paired channels, as in put_chunk
      __syncwarp();
#pragma unroll
      for (int c = 0; c < C; ++c) {
        uint32_t v0, v1, v2, v3;
        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3)
                     : "r"(src + z0_base_of(c, C) + (ch_paired(c, C) ? (dextra >> 2) : 0u)) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst + ch_base(c, C) + (ch_paired(c, C) ? dextra : 0u)), "r"(v0), "r"(v1), "r"(v2), "r"(v3) : "memory");
      }
    };
    const uint32_t park = taddr_of(tmem, 32 * q + 16, COL_R0 + 192 * h + 128);
    auto store_chunk = [&](uint32_t set, int j, const float (&v)[C][NE]) {
      uint32_t pk[C][NE];
      pack_chunk(v, pk);
      put_chunk(set, j, pk);
    };
    // One proxy fence (MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC, ~200 cycles) publishes every chunk written since the last
    // one.  The first layer's shadow path (SHP0 in bwd_layer) skips chunks 0 and 1 and publishes 0..2 with chunk_done(2).
    int chunk_pending = 0;   // first chunk written but not yet published
    auto chunk_done = [&](int j) {
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        for (int jj = chunk_pending; jj <= j; ++jj) mbar_arrive(&bar_chunk[jj]);
      }
      chunk_pending = (j + 1) & 3;
    };
    auto stash_at = [&](int l, int j, int v) { return stash + ((l * 4 + j) * NEPI * NV + v) * 32; };

    // The tensor core truncates (rounds toward zero) when it adds into an accumulator, so sums that
    // run over many tiles are kept in fp32 with round-to-nearest here: each tile's weight / bias
    // gradient accumulators start from zero and are added to this CTA's partial vector.  Every
    // element of `part` is owned by one thread, so the fire-and-forget adds are applied in tile order
    // (deterministic).  Precondition: bar_w of the tile's last step has been waited for.
    float accW[3][4][NE];  // running sums of gW_l: [layer slot][8-column block][fragment]
    float accB[3][2];      // gb_l (lanes with lane % 4 == 0 of the h == 0 warps)
    float acc0[NE];        // [gW0 | gb0] fragment (h == 0 warps)
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
      for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int e = 0; e < NE; ++e) accW[i][b][e] = 0.f;
#pragma unroll
      for (int r = 0; r < 2; ++r) accB[i][r] = 0.f;
    }
#pragma unroll
    for (int e = 0; e < NE; ++e) acc0[e] = 0.f;
    auto flush_grads = [&]() {
#pragma unroll
      for (int sl = 0; sl < 3; ++sl) {
        if (sl + 1 < n_h) {
          const uint32_t d = taddr_of(tmem, 32 * q + 16 * (sl & 1), COL_G + 64 * (sl >> 1));
          float v[4][4], w[4];
#pragma unroll
          for (int b = 0; b < 4; ++b) tmem_ld_16x256b(d + 32 * h + 8 * b, v[b]);
          tmem_ld_16x256b(taddr_of(tmem, 32 * q + 16, COL_SMALL + 8 * (sl + 1)), w);
          tmem_ld_wait();
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            float t[NE];
            pick(v[b], t);
#pragma unroll
            for (int e = 0; e < NE; ++e) accW[sl][b][e] += t[e];
          }
          float t[NE];
          pick(w, t);
#pragma unroll
          for (int r = 0; r < 2; ++r) accB[sl][r] += t[2 * r];
        }
      }
      {
        float w[4], t[NE];
        tmem_ld_16x256b(taddr_of(tmem, 32 * q + 16, COL_SMALL), w);
        tmem_ld_wait();
        pick(w, t);
#pragma unroll
        for (int e = 0; e < NE; ++e) acc0[e] += t[e];
      }
      tc_fence_before();
    };

    // point coordinates of the next tile, one (two for d = 5) per thread, fetched one tile ahead
    constexpr int XR = (TP * D + NEPI * 32 - 1) / (NEPI * 32);
    float xnext[XR];
    auto load_x = [&](int tile) {
#pragma unroll
      for (int k = 0; k < XR; ++k) {
        const int i = tid + k * NEPI * 32;
        const long long gp = (long long)tile * TP + i / D;
        xnext[k] = stream_load_if(a.X + gp * D + (i % D), pol_stream, i < TP * D && gp < a.n);
      }
    };
    if (tile_begin < tile_end) load_x(tile_begin);
    // The epilogue is at its register limit and ptxas would keep the loop bound in local memory, whose reload misses L1
    // behind the stash traffic (~1 k cycles per tile): it is kept in shared memory instead.
    if (tid == 0) *sTileEnd = tile_end;
    named_sync(1, NEPI * 32);
    auto tile_end_s = [&]() {
      int v;
      asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(sTileEnd)));
      return v;
    };
    for (int tile = tile_begin; tile < tile_end_s(); ++tile) {
      const long long base = (long long)tile * TP;
      TS(1);
      TSW(1);
      // The previous tile's first-layer MMAs may still be running: they read the adjoint set, the E tiles and the
      // OTHER x^T buffer, none of which this tile's forward sweep writes.  They are waited for in the last forward
      // layer, where their accumulators are added to the running sums.
      const uint32_t sXTb = sXT + ((tile & 1) << 11);
      named_sync(1, NEPI * 32);   // everyone is done with sX / sNb / sRed of the previous tile
      TS(3);
#pragma unroll
      for (int k = 0; k < XR; ++k)
        if (tid + k * NEPI * 32 < TP * D) sX[tid + k * NEPI * 32] = xnext[k];
      named_sync(1, NEPI * 32);
      TS(4);
      // the next tile's coordinates and this tile's coefficients are fetched now and used much later
      if (tile + 1 < tile_end_s()) load_x(tile + 1);
      const bool in_tile = tid < TP && base + tid < a.n;
      const float fv = stream_load_if(a.f ? a.f + base + tid : nullptr, pol_stream, in_tile && a.f != nullptr);
      const float bt_raw = stream_load_if(a.beta ? a.beta + base + tid : nullptr, pol_stream, in_tile && a.beta != nullptr);
      if (do_bwd) {
        for (int i = tid; i < D * 32; i += NEPI * 32) {
          const int j = i / 32, pp = 2 * (i % 32);   // row j of X^T, points pp, pp+1
          uint32_t hi, lo;
          split2(sX[pp * D + j], sX[(pp + 1) * D + j], hi, lo);
          const uint32_t off = tile_off(j, pp >> 3) + ((pp & 7) << 1);
          sts32(sXTb + off, hi);
          sts32(sXTb + 1024 + off, lo);
        }
      }

      TS(5);
      float outacc[2][C];
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) outacc[r][c] = 0.f;

      // ================= forward =================
      auto fwd_layer = [&](auto l0_tag, auto last_tag, const int l) {
        constexpr bool L0 = decltype(l0_tag)::value, LAST = decltype(last_tag)::value;
        TS(10 + l);
        if constexpr (LAST) {
          // the previous tile's gradient accumulators: nothing writes them before this tile's reverse sweep,
          // and the wait for this layer's GEMM below would be idle time otherwise
          if (w_pending) {
            mbar_wait(bar_w, ph_w);
            ph_w ^= 1;
            w_pending = false;
            tc_fence_after();
            flush_grads();
          }
        }
        if constexpr (!L0) {
          if constexpr (!SPLIT) {
            // the envelope's jet at this thread's point, while the first hidden GEMM finishes; it sits in the
            // cotangent slots (free until the residual stage, which overwrites them with the cotangents)
            if (l == 1 && a.mode == 0 && tid < TP) envelope_point<D, ORDER>(a, sX + tid * D, sNb + tid * C);
          }
          mbar_wait(bar_d, ph_d);
          ph_d ^= 1;
          tc_fence_after();
        }
        TS(20 + l);
        float xr[2][D > 0 ? D : 1];   // first layer: this thread's point coordinates (loop-invariant)
        if constexpr (L0) {
#pragma unroll
          for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int jd = 0; jd < D; ++jd) xr[r][jd] = sX[rows[r] * D + jd];
        }
        float zr[C][4];  // raw accumulator fragments [channel][ (r0,u0) (r0,u0+1) (r1,u0) (r1,u0+1) ]; chunk j+1 is fetched while chunk j is processed
        float z[C][NE];  // this thread's elements
        const uint32_t zsrc = d_addr(reg, 0) + ((32 * q) << 16) + 8 * h;
        if constexpr (!L0) {
#pragma unroll
          for (int c = 0; c < C; ++c) tmem_ld_16x256b(zsrc + ((16 * (c & 1)) << 16) + 64 * (c >> 1), zr[c]);
        }
#pragma unroll 2
        for (int j = 0; j < 4; ++j) {
          const int u0 = 16 * j + 8 * h + cq;   // this thread's columns u0, u0+1
          if constexpr (L0) {
#pragma unroll
            for (int e = 0; e < NE; ++e) {
              const int u = u0 + (e & 1);
              float v = sB[u];
#pragma unroll
              for (int jd = 0; jd < D; ++jd) v = fmaf(sW0t[jd * 64 + u], xr[e >> 1][jd], v);
              z[0][e] = v;
#pragma unroll
              for (int i = 0; i < ND; ++i) z[1 + i][e] = sW0t[(dir0 + i) * 64 + u];
              if constexpr (LAP) z[1 + ND][e] = 0.f;
            }
          } else {
            if (l == 1) TS(300 + j);
            const float b0v = sB[l * 64 + u0], b1v = sB[l * 64 + u0 + 1];   // before the wait: its "memory" clobber pins loads
            tmem_ld_wait();
            if (l == 1) TS(310 + j);
#pragma unroll
            for (int c = 0; c < C; ++c) pick_ch(zr, c, z[c]);
#pragma unroll
            for (int e = 0; e < NE; ++e) z[0][e] += (e & 1) ? b1v : b0v;
          }
          // Stash stores first: by the time the chunk's proxy fence (whose MEMBAR waits for outstanding
          // stores) is reached they have been acknowledged, and their source registers are free again.
          if (do_bwd) {
            if constexpr (!L0) {
#pragma unroll
              for (int c = 1; c < C; ++c) stash_store(stash_at(l, j, 1 + c), from_arr(z[c]), pol_stash);
            }
          }
          float av[C][NE], sv0[NE], sv1[NE];
          float zmax = 0.f;
#pragma unroll
          for (int e = 0; e < NE; ++e) zmax = fmaxf(zmax, fabsf(z[0][e]));
          const bool big = (act == 0) && __any_sync(0xffffffffu, zmax > 32768.f);
          act_eval<NE>(act, z[0], big, sv0, sv1);
          if (do_bwd) {
            stash_store(stash_at(l, j, 0), from_arr(sv0), pol_stash);
            stash_store(stash_at(l, j, 1), from_arr(sv1), pol_stash);
          }
          if constexpr (ND >= 1) {
            // chain rule on element pairs in packed fp32 arithmetic
#pragma unroll
            for (int e = 0; e < NE; e += 2) {
              float s0a, s1a, s2a, s3a, s0b, s1b, s2b, s3b;
              act_from_stash(act, sv0[e], sv1[e], s0a, s1a, s2a, s3a);
              act_from_stash(act, sv0[e + 1], sv1[e + 1], s0b, s1b, s2b, s3b);
              av[0][e] = s0a; av[0][e + 1] = s0b;
              const f32x2 S1 = pk2(s1a, s1b);
              f32x2 S;
#pragma unroll
              for (int i = 0; i < ND; ++i) {
                const f32x2 Z = pk2(z[1 + i][e], z[1 + i][e + 1]);
                unpk2(mul2(S1, Z), av[1 + i][e], av[1 + i][e + 1]);
                S = (i == 0) ? mul2(Z, Z) : fma2(Z, Z, S);
              }
              if constexpr (LAP)
                unpk2(fma2(S1, pk2(z[1 + ND][e], z[1 + ND][e + 1]), mul2(pk2(s2a, s2b), S)), av[1 + ND][e], av[1 + ND][e + 1]);
            }
          } else {
#pragma unroll
            for (int e = 0; e < NE; ++e) {
              float s0, s1, s2, s3;
              act_from_stash(act, sv0[e], sv1[e], s0, s1, s2, s3);
              av[0][e] = s0;
              float S = 0.f;
#pragma unroll
              for (int i = 0; i < ND; ++i) {
                av[1 + i][e] = s1 * z[1 + i][e];
                S = fmaf(z[1 + i][e], z[1 + i][e], S);
              }
              if constexpr (LAP) av[1 + ND][e] = fmaf(s1, z[1 + ND][e], s2 * S);
            }
          }
          if (!L0 && j < 3) {
            // z has been consumed by the chain rule: the accumulators of the next chunk are fetched under this
            // chunk's operand stores and proxy fence
#pragma unroll
            for (int c = 0; c < C; ++c) tmem_ld_16x256b(zsrc + ((16 * (c & 1)) << 16) + 64 * (c >> 1) + 16 * (j + 1), zr[c]);
          }
          if constexpr (!LAST) {
            if (l == 1) TS(320 + j);
            store_chunk(sT1, j, av);
            if (l == 1) TS(330 + j);
            chunk_done(j);
            if (l == 1) TS(340 + j);
          } else {
            const float w0v = sWL[u0], w1v = sWL[u0 + 1];
#pragma unroll
            for (int c = 0; c < C; ++c) {
#pragma unroll
              for (int r = 0; r < 2; ++r) outacc[r][c] = fmaf(w0v, av[c][2 * r], fmaf(w1v, av[c][2 * r + 1], outacc[r][c]));
            }
          }
        }
        if constexpr (!L0) reg ^= 1;
      };
      fwd_layer(std::true_type{}, std::false_type{}, 0);
      for (int l = 1; l < n_h - 1; ++l) fwd_layer(std::false_type{}, std::false_type{}, l);
      fwd_layer(std::false_type{}, std::true_type{}, n_h - 1);

      // ================= output layer + envelope + residual program =================
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
          float v = outacc[r][c];
          v += __shfl_xor_sync(0xffffffffu, v, 1);
          v += __shfl_xor_sync(0xffffffffu, v, 2);
          outacc[r][c] = v;
        }
      if ((lane & 3) == 0) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
#pragma unroll
          for (int r = 0; r < 2; ++r) sRed[(h * 64 + rows[r]) * C + c] = outacc[r][c];
        }
      }
      TSW(2);
      named_sync(1, NEPI * 32);
      float nj[C];
      if (tid < TP) {
        const long long gp = base + tid;
#pragma unroll
        for (int c = 0; c < C; ++c) nj[c] = sRed[tid * C + c] + sRed[(64 + tid) * C + c];
        nj[0] += sWL[64];
        bool programmed = false;
        if constexpr (ORDER <= 1 || SPLIT) {
          // jet modes (pde_jets_forward / pde_jets_backward): for order <= 1 the kernel's channels are the ABI's; the
          // dimension-split passes exchange (value, NDIR derivatives, partial Laplacian)
          if (a.mode == 1) {
            if (gp < a.n) {
#pragma unroll
              for (int c = 0; c < C; ++c) a.J[gp * C + c] = nj[c];
            }
            programmed = true;
          } else if (a.mode == 2) {
#pragma unroll
            for (int c = 0; c < C; ++c) nj[c] = (gp < a.n) ? a.Jbar[gp * C + c] : 0.f;
            programmed = true;
          }
        }
        if (!programmed) {
          if constexpr (!SPLIT && PARK_Q) {
            double tq[4], tg;
            q_load(tq, tg);
            if (gp < a.n) {
              program_point_lap<D, ORDER>(a, sNb + tid * C, sWL + 65, fv, a.beta ? bt_raw : a.beta_const, gp, nj, tq, tg);
            } else {
#pragma unroll
              for (int c = 0; c < C; ++c) nj[c] = 0.f;
            }
            q_store(tq, tg);
          } else if constexpr (!SPLIT) {
            if (gp < a.n) {
              program_point_lap<D, ORDER>(a, sNb + tid * C, sWL + 65, fv, a.beta ? bt_raw : a.beta_const, gp, nj, qs, gE);
            } else {
#pragma unroll
              for (int c = 0; c < C; ++c) nj[c] = 0.f;
            }
          } else {
#pragma unroll
            for (int c = 0; c < C; ++c) nj[c] = 0.f;   // split instantiations run in the jet modes only
          }
        }
      }
      TS(2);
      if (!do_bwd) continue;
      // Power-of-two scale of the adjoints, re-derived from every tile's largest network-jet cotangent and kept
      // while that maximum times the scale stays inside [2^-4, 2^8]: the 16-bit operand splits of the reverse
      // sweep then sit well inside the fp16 range whatever the size of the residual and however it drifts over
      // the CTA's tiles.  When the scale has to move, the running fp32 gradient sums are multiplied by the exact
      // power-of-two ratio (the previous tile's TMEM accumulators were flushed into them during this tile's last
      // forward layer), so the sums always carry the current scale; it is undone when the gradients are written.
      {
        float mx = 0.f;
        if (tid < TP) {
#pragma unroll
          for (int c = 0; c < C; ++c) {
            mx = fmaxf(mx, fabsf(nj[c]));
            sNb[tid * C + c] = nj[c];
          }
          // non-negative floats order like their bit patterns: one REDUX instead of a five-step shuffle tree
          mx = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(mx)));
          if (lane == 0) sMx[warp] = mx;
        }
        TSW(3);
        named_sync(1, NEPI * 32);
        TSW(4);
        mx = fmaxf(sMx[0], sMx[1]);
        const float sm = adj_scale * mx;
        if (mx > 1e-30f && mx < 3.0e38f && (adj_scale == 0.f || sm > 256.f || sm < 0.0625f)) {
          int ex = (int)((__float_as_uint(mx) >> 23) & 255u) - 126;       // mx = m 2^ex, m in [0.5, 1)
          ex = max(-60, min(60, ex));
          const float ns = __uint_as_float((uint32_t)(127 + 2 - ex) << 23);   // largest cotangent -> [2, 4)
          if (adj_scale != 0.f) {
            const float ratio = ns / adj_scale;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
              for (int b = 0; b < 4; ++b)
#pragma unroll
                for (int e = 0; e < NE; ++e) accW[i][b][e] *= ratio;
#pragma unroll
              for (int r = 0; r < 2; ++r) accB[i][r] *= ratio;
            }
#pragma unroll
            for (int e = 0; e < NE; ++e) acc0[e] *= ratio;
#pragma unroll
            for (int j = 0; j < 4; ++j) { gwl[j][0] *= ratio; gwl[j][1] *= ratio; }
            gbl *= ratio;
          }
          adj_scale = ns;
        }
        cur_scale = (adj_scale != 0.f) ? adj_scale : 1.f;   // all cotangents so far are zero: nothing to scale
        if (tid < TP) gbl += nj[0] * cur_scale;
      }

      // ================= reverse sweep =================
      auto bwd_layer = [&](auto top_tag, auto lk_tag, const int l) {
        constexpr bool TOP = decltype(top_tag)::value;
        constexpr int LK = decltype(lk_tag)::value;   // 0: first layer, 1: l == 1, 2: l >= 2
        // Stash of this layer (activation values, pre-activation jets) and of the layer below (whose
        // activations are this layer's wgrad operand).  Software pipeline: the registers of chunk j+1
        // are fetched as soon as chunk j has consumed them (no rotation copies).
        float4 cur[NV], prv[NV];
        auto load_cur = [&](int j) {
          cur[0] = stash_load(stash_at(l, j, 0), pol_stash); cur[1] = stash_load(stash_at(l, j, 1), pol_stash);
          if constexpr (LK >= 1) {
#pragma unroll
            for (int v = 2; v < NV; ++v) cur[v] = stash_load(stash_at(l, j, v), pol_stash);
          }
        };
        // at the top layer A_{n_h-2} is still in T1 from the forward sweep: nothing to rebuild
        constexpr bool REFILL = (LK >= 1) && !TOP;
        auto load_prv = [&](int j) {
          if constexpr (REFILL) {
            prv[0] = stash_load(stash_at(l - 1, j, 0), pol_stash); prv[1] = stash_load(stash_at(l - 1, j, 1), pol_stash);
            if constexpr (LK >= 2) {
#pragma unroll
              for (int v = 2; v < NV; ++v) prv[v] = stash_load(stash_at(l - 1, j, v), pol_stash);
            }
          }
        };
        // Shadow builds, below the top layer (SH): chunk 0 of the adjoints goes to the shadow, so nothing waits for
        // the previous layer's wgrad before chunk 1; chunk 0 of the rebuilt A_{l-1} is parked in TMEM until the sets
        // are free.
        constexpr bool SH = SHADOW && !TOP;
        load_cur(0);
        load_prv(0);
        TS(30 + l);
        if constexpr (!TOP) {
          mbar_wait(bar_d, ph_d);   // Ab_l is complete
          ph_d ^= 1;
          tc_fence_after();
        }
        TS(40 + l);
        float nbr[2][C];   // top layer: cotangents of this thread's points (loop-invariant)
        if constexpr (TOP) {
#pragma unroll
          for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c) nbr[r][c] = sNb[rows[r] * C + c] * cur_scale;
        }
        float abr[C][4];   // raw accumulator fragments
        float ab[C][NE];
        const uint32_t absrc = d_addr(reg, 0) + ((32 * q) << 16) + 8 * h;
        if constexpr (!TOP) {
#pragma unroll
          for (int c = 0; c < C; ++c) tmem_ld_16x256b(absrc + ((16 * (c & 1)) << 16) + 64 * (c >> 1), abr[c]);
        }
        auto refill = [&](const int u0, float (&ap)[C][NE]) {
          // activations of layer l-1 (operand of this layer's wgrad) recomputed from its stash
          float pv0[NE], pv1[NE];
          to_arr(prv[0], pv0);
          to_arr(prv[1], pv1);
          float zp[C][NE];
          if constexpr (LK >= 2) {
#pragma unroll
            for (int c = 1; c < C; ++c) to_arr(prv[1 + c], zp[c]);
          } else {
#pragma unroll
            for (int e = 0; e < NE; ++e) {
              const int u = u0 + (e & 1);
#pragma unroll
              for (int i = 0; i < ND; ++i) zp[1 + i][e] = sW0t[(dir0 + i) * 64 + u];
              if constexpr (LAP) zp[1 + ND][e] = 0.f;
            }
          }
          if constexpr (ND >= 1) {
#pragma unroll
            for (int e = 0; e < NE; e += 2) {
              float s0a, s1a, s2a, s3a, s0b, s1b, s2b, s3b;
              act_from_stash(act, pv0[e], pv1[e], s0a, s1a, s2a, s3a);
              act_from_stash(act, pv0[e + 1], pv1[e + 1], s0b, s1b, s2b, s3b);
              ap[0][e] = s0a; ap[0][e + 1] = s0b;
              const f32x2 S1 = pk2(s1a, s1b);
              f32x2 S = 0;
#pragma unroll
              for (int i = 0; i < ND; ++i) {
                const f32x2 Z = pk2(zp[1 + i][e], zp[1 + i][e + 1]);
                unpk2(mul2(S1, Z), ap[1 + i][e], ap[1 + i][e + 1]);
                S = (i == 0) ? mul2(Z, Z) : fma2(Z, Z, S);
              }
              if constexpr (LAP)
                unpk2(fma2(S1, pk2(zp[1 + ND][e], zp[1 + ND][e + 1]), mul2(pk2(s2a, s2b), S)), ap[1 + ND][e], ap[1 + ND][e + 1]);
            }
          } else {
#pragma unroll
            for (int e = 0; e < NE; ++e) {
              float s0, s1, s2, s3;
              act_from_stash(act, pv0[e], pv1[e], s0, s1, s2, s3);
              ap[0][e] = s0;
              float S = 0.f;
#pragma unroll
              for (int i = 0; i < ND; ++i) {
                ap[1 + i][e] = s1 * zp[1 + i][e];
                S = fmaf(zp[1 + i][e], zp[1 + i][e], S);
              }
              if constexpr (LAP) ap[1 + ND][e] = fmaf(s1, zp[1 + ND][e], s2 * S);
            }
          }
        };
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {
          const int u0 = 16 * j + 8 * h + cq;
          uint32_t zk[C][NE];
          {
          if constexpr (TOP) {
            const float w0v = sWL[u0], w1v = sWL[u0 + 1];
#pragma unroll
            for (int c = 0; c < C; ++c) {
#pragma unroll
              for (int r = 0; r < 2; ++r) {
                const float nv = nbr[r][c];
                ab[c][2 * r] = w0v * nv; ab[c][2 * r + 1] = w1v * nv;
              }
            }
          } else {
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < C; ++c) pick_ch(abr, c, ab[c]);
          }
          float zb[C][NE];
          {
            float sv0[NE], sv1[NE];
            to_arr(cur[0], sv0);
            to_arr(cur[1], sv1);
            float zj[C][NE];   // zj[1..]: derivative channels of z (zj[0] unused)
            if constexpr (LK >= 1) {
#pragma unroll
              for (int c = 1; c < C; ++c) to_arr(cur[1 + c], zj[c]);
            } else {
#pragma unroll
              for (int e = 0; e < NE; ++e) {
                const int u = u0 + (e & 1);
#pragma unroll
                for (int i = 0; i < ND; ++i) zj[1 + i][e] = sW0t[(dir0 + i) * 64 + u];
                if constexpr (LAP) zj[1 + ND][e] = 0.f;
              }
            }
            if constexpr (ND >= 1) {
              // the same recurrences on element pairs in packed fp32 arithmetic
#pragma unroll
              for (int e = 0; e < NE; e += 2) {
                float s0a, s1a, s2a, s3a, s0b, s1b, s2b, s3b;
                act_from_stash(act, sv0[e], sv1[e], s0a, s1a, s2a, s3a);
                act_from_stash(act, sv0[e + 1], sv1[e + 1], s0b, s1b, s2b, s3b);
                const f32x2 S1 = pk2(s1a, s1b), S2 = pk2(s2a, s2b);
                f32x2 T0 = mul2(S1, pk2(ab[0][e], ab[0][e + 1]));
                f32x2 ABL = 0, S = 0;
                if constexpr (LAP) ABL = pk2(ab[1 + ND][e], ab[1 + ND][e + 1]);
#pragma unroll
                for (int i = 0; i < ND; ++i) {
                  const f32x2 Z = pk2(zj[1 + i][e], zj[1 + i][e + 1]);
                  const f32x2 AB = pk2(ab[1 + i][e], ab[1 + i][e + 1]);
                  const f32x2 S2Z = mul2(S2, Z);
                  T0 = fma2(S2Z, AB, T0);
                  S = (i == 0) ? mul2(Z, Z) : fma2(Z, Z, S);
                  f32x2 Ti = mul2(S1, AB);
                  if constexpr (LAP) Ti = fma2(add2(S2Z, S2Z), ABL, Ti);
                  unpk2(Ti, zb[1 + i][e], zb[1 + i][e + 1]);
                }
                if constexpr (LAP) {
                  T0 = fma2(fma2(S2, pk2(zj[1 + ND][e], zj[1 + ND][e + 1]), mul2(pk2(s3a, s3b), S)), ABL, T0);
                  unpk2(mul2(S1, ABL), zb[1 + ND][e], zb[1 + ND][e + 1]);
                }
                unpk2(T0, zb[0][e], zb[0][e + 1]);
                if constexpr (TOP) {
                  // output-layer weight gradient: sum_c nb_c a_c with a_c recomputed from the stash
                  float Sa, Sb;
                  unpk2(S, Sa, Sb);
                  const int r = e >> 1;
                  float ga = nbr[r][0] * s0a, gb = nbr[r][0] * s0b;
#pragma unroll
                  for (int i = 0; i < ND; ++i) {
                    ga = fmaf(nbr[r][1 + i], s1a * zj[1 + i][e], ga);
                    gb = fmaf(nbr[r][1 + i], s1b * zj[1 + i][e + 1], gb);
                  }
                  if constexpr (LAP) {
                    ga = fmaf(nbr[r][1 + ND], fmaf(s1a, zj[1 + ND][e], s2a * Sa), ga);
                    gb = fmaf(nbr[r][1 + ND], fmaf(s1b, zj[1 + ND][e + 1], s2b * Sb), gb);
                  }
                  gwl[j][0] += ga;
                  gwl[j][1] += gb;
                }
              }
            } else {
  #pragma unroll
              for (int e = 0; e < NE; ++e) {
                float s0, s1, s2, s3;
                act_from_stash(act, sv0[e], sv1[e], s0, s1, s2, s3);
                float t0 = s1 * ab[0][e];
                float abL = 0.f;
                if constexpr (LAP) abL = ab[1 + ND][e];
                float S = 0.f;
  #pragma unroll
                for (int i = 0; i < ND; ++i) {
                  const float zi = zj[1 + i][e];
                  t0 = fmaf(s2 * zi, ab[1 + i][e], t0);
                  S = fmaf(zi, zi, S);
                  float ti = s1 * ab[1 + i][e];
                  if constexpr (LAP) ti = fmaf(2.f * s2 * zi, abL, ti);
                  zb[1 + i][e] = ti;
                }
                if constexpr (LAP) {
                  t0 = fmaf(fmaf(s2, zj[1 + ND][e], s3 * S), abL, t0);
                  zb[1 + ND][e] = s1 * abL;
                }
                zb[0][e] = t0;
                if constexpr (TOP) {
                  // output-layer weight gradient: sum_c nb_c a_c with a_c recomputed from the stash
                  const int r = e >> 1;
                  float g = nbr[r][0] * s0;
  #pragma unroll
                  for (int i = 0; i < ND; ++i) g = fmaf(nbr[r][1 + i], s1 * zj[1 + i][e], g);
                  if constexpr (LAP) g = fmaf(nbr[r][1 + ND], fmaf(s1, zj[1 + ND][e], s2 * S), g);
                  gwl[j][e & 1] += g;
                }
              }
                      }
}
          if (j < 3) {
            // ab and cur have been consumed: fetch chunk j+1
            if constexpr (!TOP) {
#pragma unroll
              for (int c = 0; c < C; ++c) tmem_ld_16x256b(absrc + ((16 * (c & 1)) << 16) + 64 * (c >> 1) + 16 * (j + 1), abr[c]);
            }
            load_cur(j + 1);
          }
          pack_chunk(zb, zk);
          }
          float ap[C][NE];
          if (REFILL) {
            refill(u0, ap);
            if (j < 3) load_prv(j + 1);
          }
          // first layer (no GEMM consumes its chunks one by one): chunk 1 is parked as well and the wait moves to chunk 2
          constexpr bool SHP0 = SH && LK == 0;
          if (j == (SH ? (SHP0 ? 2 : 1) : 0) && w_pending) {
            // the previous layer's wgrad still reads both operand sets: the results of this chunk are
            // computed before waiting for it, the stores come after
            TS(50 + l);
            mbar_wait(bar_w, ph_w);
            ph_w ^= 1;
            w_pending = false;
            TS(60 + l);
          }
          if constexpr (SHP0) {
            if (j <= 2) {
              if (j == 0) {
                put_shadow(zk);
              } else if (j == 1) {
#pragma unroll
                for (int c = 0; c < C; ++c) tmem_st_16x256b_u32(park + 8 * c, zk[c]);
                tmem_st_wait();
              } else {
                put_chunk(sT2, 2, zk);
                uint32_t pk[C][NE];
#pragma unroll
                for (int c = 0; c < C; ++c) tmem_ld_16x256b_u32(park + 8 * c, pk[c]);
                tmem_ld_wait();
                put_chunk(sT2, 1, pk);
                copy_shadow();
                chunk_done(2);   // publishes chunks 0..2
              }
              continue;
            }
          }
          if (SH && j == 0) {
            put_shadow(zk);
            if constexpr (REFILL) {
              // park the split A_{l-1} chunk in the unused accumulator slot of region h (lane half 1, columns 128..)
              uint32_t pk[C][NE];
              pack_chunk(ap, pk);
#pragma unroll
              for (int c = 0; c < C; ++c) tmem_st_16x256b_u32(park + 8 * c, pk[c]);
              tmem_st_wait();
            }
          } else {
            put_chunk(sT2, j, zk);
            if constexpr (REFILL) store_chunk(sT1, j, ap);
            if constexpr (SH) if (j == 1) {
              // the sets are free: chunk 0 moves from the shadow / TMEM to its place
              if constexpr (REFILL) {
                uint32_t pk[C][NE];
#pragma unroll
                for (int c = 0; c < C; ++c) tmem_ld_16x256b_u32(park + 8 * c, pk[c]);
                tmem_ld_wait();
                put_chunk(sT1, 0, pk);
              }
              copy_shadow();
            }
          }
          chunk_done(j);
        }
        if constexpr (!TOP) reg ^= 1;
        w_pending = true;   // the issuer commits bar_w after this step's wgrad / first-layer MMAs
      };
      using I0 = std::integral_constant<int, 0>;
      using I1 = std::integral_constant<int, 1>;
      using I2 = std::integral_constant<int, 2>;
      if (n_h - 1 >= 2) bwd_layer(std::true_type{}, I2{}, n_h - 1);
      else bwd_layer(std::true_type{}, I1{}, n_h - 1);
      for (int l = n_h - 2; l >= 2; --l) bwd_layer(std::false_type{}, I2{}, l);
      if (n_h - 2 >= 1) bwd_layer(std::false_type{}, I1{}, 1);
      bwd_layer(std::false_type{}, I0{}, 0);
    }

    // ================= per-CTA results =================
    if (w_pending) {
      mbar_wait(bar_w, ph_w);
      ph_w ^= 1;
      tc_fence_after();
      flush_grads();
    }
    if (do_bwd) {
      const float inv = (adj_scale != 0.f) ? 1.f / adj_scale : 1.f;   // exact: a power of two
      // hidden GEMM layers: gW_l at slot l-1, rows o = 16 q + lane/4 (+8), columns i
#pragma unroll
      for (int sl = 0; sl < 3; ++sl) {
        if (sl + 1 < n_h) {
          float* gW = part + a.off_gW + (long long)sl * ((long long)HP * HP + HP);
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const int i0 = 32 * h + 8 * b + cq;
#pragma unroll
            for (int r = 0; r < 2; ++r)
              *reinterpret_cast<float2*>(gW + rows[r] * HP + i0) = make_float2(accW[sl][b][2 * r] * inv, accW[sl][b][2 * r + 1] * inv);
          }
          if (h == 0 && (lane & 3) == 0) {
#pragma unroll
            for (int r = 0; r < 2; ++r) gW[HP * HP + rows[r]] = accB[sl][r] * inv;
          }
        }
      }
      if (h == 0) {
        // columns cq, cq+1 of [gW0 (D cols) | gb0]
#pragma unroll
        for (int e = 0; e < NE; ++e) {
          const int col = cq + (e & 1), o = rows[e >> 1];
          if (col < D) part[a.off_gW0 + o * D + col] = acc0[e] * inv;
          else if (col == D) part[a.off_gb0 + o] = acc0[e] * inv;
        }
      }
      // output layer: reduce the per-thread column partials over the 8 row groups of the warp ...
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          float v = gwl[j][k];
          v += __shfl_xor_sync(0xffffffffu, v, 4);
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          gwl[j][k] = v;
        }
      named_sync(1, NEPI * 32);
      float* sRedW = sRed;   // [4 row groups][64 columns]
      if (lane < 4) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          sRedW[q * 64 + 16 * j + 8 * h + cq] = gwl[j][0];
          sRedW[q * 64 + 16 * j + 8 * h + cq + 1] = gwl[j][1];
        }
      }
      named_sync(1, NEPI * 32);
      // ... then over the row groups in fixed order
      if (tid < 64) {
        const float v = (sRedW[tid] + sRedW[64 + tid]) + (sRedW[128 + tid] + sRedW[192 + tid]);
        part[a.off_gwL + tid] = v * inv;
      }
      named_sync(1, NEPI * 32);
      if (tid < 64) sRed[tid] = gbl;
      named_sync(1, NEPI * 32);
      if (tid == 0) {
        float v = 0.f;
        for (int i = 0; i < 64; ++i) v += sRed[i];
        part[a.off_gbL] = v * inv;
      }
    }
    named_sync(1, NEPI * 32);
    {
      double* dred = reinterpret_cast<double*>(sm + SM::off_T1);   // 64 x 5 doubles
      if (tid < TP) {
        if constexpr (PARK_Q) q_load(qs, gE);
#pragma unroll
        for (int k = 0; k < 4; ++k) dred[tid * 5 + k] = qs[k];
        dred[tid * 5 + 4] = gE;
      }
      named_sync(1, NEPI * 32);
      if (tid < 5) {
        double v = 0.0;
        for (int pp = 0; pp < TP; ++pp) v += dred[pp * 5 + tid];
        a.psums[(long long)blockIdx.x * 8 + tid] = v;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------- 5-D PINN: residual stage between the two split passes
// Per point: network jets of the two dimension-split forward passes (J_A: value, d_0..d_2, Lap over dims 0..2;
// J_B: value, d_3, d_4, Lap over dims 3..4) -> envelope, residual program and per-point seeds exactly as in the fused
// kernel (program_point_lap on (value, 5 derivatives, full Laplacian)) -> cotangents of both passes.  HBM-bound:
// 4 (5 + 2 + 9 + 9) bytes per point, coalesced, grid = 4 x SMs.
__global__ void pinn_split_kernel(const TcArgs a, const float* JA, const float* JB, float* JbarA, float* JbarB, double* psums) {
  double qs[4] = {0.0, 0.0, 0.0, 0.0};
  double gE = 0.0;
  const float cst[3] = {a.energy ? a.energy[0] : a.energy_const, (a.seed ? a.seed[0] : 1.f) * a.inv_n,
                        (a.seed && a.prog == PDE_PROG_RAYLEIGH ? a.seed[1] : 1.f) * a.inv_n};
  for (long long gp = blockIdx.x * (long long)blockDim.x + threadIdx.x; gp < a.n; gp += (long long)gridDim.x * blockDim.x) {
    float x[5], nj[7];
#pragma unroll
    for (int i = 0; i < 5; ++i) x[i] = a.X[gp * 5 + i];
    nj[0] = JA[gp * 5];
    nj[1] = JA[gp * 5 + 1]; nj[2] = JA[gp * 5 + 2]; nj[3] = JA[gp * 5 + 3];
    nj[4] = JB[gp * 4 + 1]; nj[5] = JB[gp * 4 + 2];
    nj[6] = JA[gp * 5 + 4] + JB[gp * 4 + 3];
    const float fv = a.f ? a.f[gp] : 0.f;
    const float bt = a.beta ? a.beta[gp] : a.beta_const;
    float env[7];
    envelope_point<5, 2>(a, x, env);
    program_point_lap<5, 2>(a, env, cst, fv, bt, gp, nj, qs, gE);
    if (JbarA) {
      // the value channel's cotangent goes to pass A only (the reverse sweep is linear in the cotangents)
      JbarA[gp * 5] = nj[0]; JbarA[gp * 5 + 1] = nj[1]; JbarA[gp * 5 + 2] = nj[2]; JbarA[gp * 5 + 3] = nj[3]; JbarA[gp * 5 + 4] = nj[6];
      JbarB[gp * 4] = 0.f; JbarB[gp * 4 + 1] = nj[4]; JbarB[gp * 4 + 2] = nj[5]; JbarB[gp * 4 + 3] = nj[6];
    }
  }
  __shared__ double sh[8][5];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    double v = (k < 4) ? qs[k] : gE;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) sh[wid][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    double v = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) v += sh[i][threadIdx.x];
    psums[(long long)blockIdx.x * 8 + threadIdx.x] = v;
  }
}

// ---------------------------------------------------------------- parameter images
struct TcPackArgs {
  const float* W[PDE_MAX_LINEAR];
  const float* b[PDE_MAX_LINEAR];
  int n_lin, D, H;
  float* params;           // W0t [D][64], b [n_h][64], wL [64], bL
  unsigned char* wimg;     // [(n_h-1)][2][8192]
};

__global__ void tc_pack_kernel(const TcPackArgs a) {
  const int n_h = a.n_lin - 1;
  const int n_par = a.D * 64 + n_h * 64 + 64 + 1;
  const int n_img = (n_h - 1) * 64 * 32;   // pairs of adjacent columns
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_par + n_img; i += gridDim.x * blockDim.x) {
    if (i < n_par) {
      float v = 0.f;
      if (i < a.D * 64) {
        const int j = i / 64, u = i % 64;
        if (u < a.H) v = a.W[0][u * a.D + j];
      } else if (i < a.D * 64 + n_h * 64) {
        const int r = i - a.D * 64, l = r / 64, u = r % 64;
        if (u < a.H) v = a.b[l][u];
      } else if (i < a.D * 64 + n_h * 64 + 64) {
        const int u = i - a.D * 64 - n_h * 64;
        if (u < a.H) v = a.W[n_h][u];
      } else {
        v = a.b[n_h][0];
      }
      a.params[i] = v;
    } else {
      const int r = i - n_par, l = r / (64 * 32) + 1, e = r % (64 * 32), o = e / 32, i0 = 2 * (e % 32);
      float x0 = 0.f, x1 = 0.f;
      if (o < a.H) {
        if (i0 < a.H) x0 = a.W[l][o * a.H + i0];
        if (i0 + 1 < a.H) x1 = a.W[l][o * a.H + i0 + 1];
      }
      uint32_t hi, lo;
      split2(x0, x1, hi, lo);
      unsigned char* img = a.wimg + (size_t)(l - 1) * 2 * TILE_BYTES;
      const uint32_t off = tile_off(o, i0 >> 3) + ((i0 & 7) << 1);
      *reinterpret_cast<uint32_t*>(img + off) = hi;
      *reinterpret_cast<uint32_t*>(img + TILE_BYTES + off) = lo;
    }
  }
}

// ---------------------------------------------------------------- host side
struct TcPlan {
  int D, order, C, NV, n_lin, n_h, H, grid, num_tiles, sms;
  int ndir;   // derivative directions of this launch (= D except in the dimension-split passes)
  size_t smem_bytes;
  GradLayout g;
  long long stash_f4;
  size_t ws_params, ws_wimg, ws_partial, ws_psums, ws_stash, ws_total;
};

template <int D, int ORDER, int ACT, int NDIR = D>
static cudaError_t launch_one(const TcPlan& p, const TcArgs& a, cudaStream_t st) {
  constexpr int C = 1 + (ORDER >= 1 ? NDIR : 0) + (ORDER == 2);
  if constexpr (C > MAXC) {
    return cudaErrorInvalidValue;
  } else {
    const int smem = SmemMap<D, C>::total;
    cudaError_t err = cudaFuncSetAttribute(tc_kernel<D, ORDER, ACT, NDIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess) return err;
    tc_kernel<D, ORDER, ACT, NDIR><<<p.grid, NTHREADS, smem, st>>>(a);
    return cudaGetLastError();
  }
}

template <int ACT>
static cudaError_t launch_act(const TcPlan& p, const TcArgs& a, cudaStream_t st) {
  if (p.ndir != p.D) {   // dimension-split passes of the 5-D PINN step
#if !defined(PDE_TC_ONLY_CFG2) && !defined(PDE_TC_ONLY_SMALL)
    if (p.D == 5 && p.order == 2 && p.ndir == 3) return launch_one<5, 2, ACT, 3>(p, a, st);
    if (p.D == 5 && p.order == 2 && p.ndir == 2) return launch_one<5, 2, ACT, 2>(p, a, st);
#endif
    return cudaErrorInvalidValue;
  }
#ifdef PDE_TC_ONLY_CFG2   // development builds (A/B timing of kernel variants): configs 2 and 3 only
  if (p.D == 3 && p.order == 2 && ACT == 0) return launch_one<3, 2, 0>(p, a, st);
  if (p.D == 5 && p.order == 1 && ACT == 0) return launch_one<5, 1, 0>(p, a, st);
  return cudaErrorInvalidValue;
#elif defined(PDE_TC_ONLY_SMALL)   // development builds: the three-channel variants of configs 1 and 4
  if (p.D == 1 && p.order == 2 && ACT == 0) return launch_one<1, 2, 0>(p, a, st);
  if (p.D == 2 && p.order == 1 && ACT == 0) return launch_one<2, 1, 0>(p, a, st);
  if (p.D == 2 && p.order == 2 && ACT == 1) return launch_one<2, 2, 1>(p, a, st);
  return cudaErrorInvalidValue;
#else
  switch (p.D * 3 + p.order) {
    case 3: return launch_one<1, 0, ACT>(p, a, st);
    case 4: return launch_one<1, 1, ACT>(p, a, st);
    case 5: return launch_one<1, 2, ACT>(p, a, st);
    case 6: return launch_one<2, 0, ACT>(p, a, st);
    case 7: return launch_one<2, 1, ACT>(p, a, st);
    case 8: return launch_one<2, 2, ACT>(p, a, st);
    case 9: return launch_one<3, 0, ACT>(p, a, st);
    case 10: return launch_one<3, 1, ACT>(p, a, st);
    case 11: return launch_one<3, 2, ACT>(p, a, st);
    case 12: return launch_one<4, 0, ACT>(p, a, st);
    case 13: return launch_one<4, 1, ACT>(p, a, st);
    case 14: return launch_one<4, 2, ACT>(p, a, st);
    case 15: return launch_one<5, 0, ACT>(p, a, st);
    case 16: return launch_one<5, 1, ACT>(p, a, st);
    default: return cudaErrorInvalidValue;
  }
#endif
}

static cudaError_t launch_tc(const TcPlan& p, const TcArgs& a, cudaStream_t st) {
  return a.act == PDE_ACT_TANH ? launch_act<1>(p, a, st) : launch_act<0>(p, a, st);
}

// Kernel-family override: -1 automatic (tensor-core kernel where supported), 0 generic SIMT kernel, 1 tensor-core
// kernel also below its size threshold.  Initial value from PDE_B200_PATH=simt|tc, read once; pde_set_kernel_path
// changes it (parity tests run both families on the same inputs).
static std::atomic<int> g_path_override{-2};
static int path_override() {
  int v = g_path_override.load(std::memory_order_relaxed);
  if (v == -2) {
    const char* e = getenv("PDE_B200_PATH");
    v = !e ? -1 : (strcmp(e, "simt") == 0 ? 0 : (strcmp(e, "tc") == 0 ? 1 : -1));
    g_path_override.store(v, std::memory_order_relaxed);
  }
  return v;
}

#ifdef PDE_TC_TIMELINE
// Development build only (make EXTRA=-DPDE_TC_TIMELINE): PDE_B200_TIMELINE=<file> records (event, clock)
// pairs of CTA 0 and writes them after the launch (this synchronises the stream).
static long long* timeline_buffer() {
  static long long* buf = nullptr;
  if (!getenv("PDE_B200_TIMELINE")) return nullptr;
  if (!buf && cudaMalloc(&buf, 16384 * sizeof(long long)) != cudaSuccess) return nullptr;
  cudaMemset(buf, 0, 16384 * sizeof(long long));
  return buf;
}
static void timeline_dump(long long* buf, cudaStream_t st) {
  if (!buf) return;
  cudaStreamSynchronize(st);
  static long long host[16384];
  cudaMemcpy(host, buf, sizeof(host), cudaMemcpyDeviceToHost);
  FILE* f = fopen(getenv("PDE_B200_TIMELINE"), "w");
  if (!f) return;
  for (int w = 0; w < 2; ++w)
    for (int i = 0; i < 2000 && host[w * 4096 + 2 * i] != 0; ++i)
      fprintf(f, "%d %lld %lld\n", w, host[w * 4096 + 2 * i], host[w * 4096 + 2 * i + 1]);
  for (int w = 0; w < 8; ++w)
    for (int i = 0; i < 500 && host[8192 + w * 1024 + 2 * i] != 0; ++i)
      fprintf(f, "%d %lld %lld\n", 10 + w, host[8192 + w * 1024 + 2 * i], host[8192 + w * 1024 + 2 * i + 1]);
  fclose(f);
}
#endif

static bool shape_ok(const pde_net* net, int order, long long n, int ndir = -1) {
  if (!net || net->dtype != PDE_F32) return false;
  if (net->dim < 1 || net->dim > PDE_MAX_DIM) return false;
  const int n_h = net->n_linear - 1;
  if (n_h < 2 || n_h > 4) return false;
  const int H = net->widths[1];
  if (H < 1 || H > HP) return false;
  for (int l = 1; l < net->n_linear; ++l)
    if (net->widths[l] != H) return false;
  if (net->widths[0] != net->dim || net->widths[net->n_linear] != 1) return false;
  if (order < 0 || order > 2) return false;
  const int C = 1 + (order >= 1 ? (ndir < 0 ? net->dim : ndir) : 0) + (order == 2);
  if (C > MAXC) return false;
  const int ov = path_override();
  if (ov == 0) return false;
  if (ov == 1) return n >= 1;
  return n >= 4096;   // below that the launch is latency bound and the generic kernel is as fast
}

static int make_plan(const pde_net* net, int order, long long n, TcPlan* pl, int ndir = -1) {
  if (!shape_ok(net, order, n, ndir)) return PDE_ERR_UNSUPPORTED;
  const DevInfo dv = device_info();
  if (!dv.ok) return PDE_ERR_NO_DEVICE;
  if (dv.cc_major != 10) return PDE_ERR_UNSUPPORTED;
  TcPlan& p = *pl;
  memset(&p, 0, sizeof(p));
  p.sms = dv.sms;
  p.D = net->dim; p.order = order;
  p.ndir = ndir < 0 ? p.D : ndir;
  p.C = 1 + (order >= 1 ? p.ndir : 0) + (order == 2);
  p.NV = 1 + p.C;
  p.n_lin = net->n_linear; p.n_h = p.n_lin - 1; p.H = net->widths[1];
  p.num_tiles = (int)((n + TP - 1) / TP);
  p.grid = p.num_tiles < p.sms ? p.num_tiles : p.sms;
  p.g = grad_layout(p.D, p.n_h, p.H, HP);
  p.stash_f4 = (long long)p.n_h * 4 * 8 * p.NV * 32;   // 16 bytes per thread of 8 warps (or 8 bytes x 16 warps)
  p.ws_params = (size_t)rup((p.D * 64 + p.n_h * 64 + 64 + 1) * 4, 256);
  p.ws_wimg = (size_t)(p.n_h - 1) * 2 * TILE_BYTES;
  p.ws_partial = (size_t)rup((long long)p.sms * p.g.PP * 4, 256);
  p.ws_psums = (size_t)rup((long long)p.sms * 8 * 8, 256);
  p.ws_stash = (size_t)rup((long long)p.sms * p.stash_f4 * 16, 256);
  p.ws_total = p.ws_params + p.ws_wimg + p.ws_partial + p.ws_psums + p.ws_stash;
  return PDE_OK;
}

// The workspace pieces every tensor-core sequence uses, as make_plan sized them.
struct TcBufs {
  float* params;
  unsigned char* wimg;
  float* partial;
  double* psums;
  float4* stash;
};

static TcBufs carve(const TcPlan& p, void* workspace) {
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  TcBufs b;
  b.params = reinterpret_cast<float*>(wsb);
  b.wimg = wsb + p.ws_params;
  b.partial = reinterpret_cast<float*>(wsb + p.ws_params + p.ws_wimg);
  b.psums = reinterpret_cast<double*>(wsb + p.ws_params + p.ws_wimg + p.ws_partial);
  b.stash = reinterpret_cast<float4*>(wsb + p.ws_params + p.ws_wimg + p.ws_partial + p.ws_psums);
  return b;
}

static int launch_tc_pack(const pde_net* net, const TcPlan& p, float* params, unsigned char* wimg, cudaStream_t st) {
  TcPackArgs pa;
  memset(&pa, 0, sizeof(pa));
  for (int l = 0; l < p.n_lin; ++l) { pa.W[l] = static_cast<const float*>(net->W[l]); pa.b[l] = static_cast<const float*>(net->b[l]); }
  pa.n_lin = p.n_lin; pa.D = p.D; pa.H = p.H; pa.params = params; pa.wimg = wimg;
  tc_pack_kernel<<<32, 256, 0, st>>>(pa);
  if (cudaGetLastError() != cudaSuccess) return PDE_ERR_CUDA;
  count_launch();
  return PDE_OK;
}

// tc_kernel arguments of every mode: network, points, workspace and the partial-gradient layout.
static TcArgs tc_args(const pde_net* net, const TcPlan& p, const TcBufs& b, const void* X, long long n, int mode,
                      double inv_n) {
  TcArgs a;
  memset(&a, 0, sizeof(a));
  a.n_h = p.n_h; a.act = net->activation; a.H = p.H;
  a.params = b.params; a.wimg = b.wimg;
  a.X = static_cast<const float*>(X); a.n = n; a.num_tiles = p.num_tiles;
  a.mode = mode;
  a.inv_n = (float)inv_n;
  a.partial = b.partial; a.psums = b.psums; a.stash = b.stash;
  a.PP = p.g.PP; a.stash_f4 = p.stash_f4;
  a.off_gW0 = p.g.off_gW0; a.off_gb0 = p.g.off_gb0; a.off_gW = p.g.off_gW; a.off_gwL = p.g.off_gwL; a.off_gbL = p.g.off_gbL;
  return a;
}

// What the envelope and residual-program stage reads (tc_kernel in mode 0, pinn_split_kernel).
static void set_program(TcArgs& a, const pde_envelope* env, const pde_program* prog, const void* seed, double inv_n) {
  a.prog = prog->kind; a.n_q = pde_program_quantities(prog->kind);
  fill_env<float>(env, &a.env);
  a.alpha = (float)prog->alpha; a.beta_const = (float)prog->beta_const; a.energy_const = (float)prog->energy_const;
  a.inv_n = (float)inv_n;
  a.f = static_cast<const float*>(prog->f); a.beta = static_cast<const float*>(prog->beta);
  a.energy = static_cast<const float*>(prog->energy); a.seed = static_cast<const float*>(seed);
  a.faces = prog->faces; a.face_n = flux_face_n(prog, a.n);
}

}  // namespace tc

// Every residual program is served.  (Round 1 kept the Rayleigh quotient on the generic kernel: its gradient is a
// difference of nearly parallel vectors, which amplifies the ~1e-6 rounding of the split GEMMs.  Measured at the
// reference's own shapes — 200 x 200 grids, [2,50,50,50,50,1], tools/rayleigh_check.py — the tensor-core gradients are
// 1.4e-6 .. 8.9e-6 from the float64 reference, inside the bar each fixture justifies.)
static bool program_ok(const pde_program* prog) { return prog != nullptr; }

// 5-D second-order programs need 7 jet channels, one more than fits on chip: they run as two dimension-split passes
// (3 + 2 directions, 5 and 4 channels) around a pointwise residual kernel (tc_pinn_split below).
static bool split_shape(const pde_net* net, int order) { return net && net->dim == 5 && order == 2; }
constexpr int SPLIT_BLOCK = 256;
struct SplitPlan {
  tc::TcPlan a, b;          // passes over directions 0..2 and 3..4
  int blocks;               // pointwise kernel
  size_t ws_common, off_JA, off_JB, off_JbA, off_JbB, off_ps, ws_total;
};
static int make_split_plan(const pde_net* net, long long n, SplitPlan* sp) {
  int rc = tc::make_plan(net, 2, n, &sp->a, 3);
  if (rc) return rc;
  if ((rc = tc::make_plan(net, 2, n, &sp->b, 2))) return rc;
  long long g = (n + SPLIT_BLOCK - 1) / SPLIT_BLOCK;
  sp->blocks = (int)(g < 4LL * sp->a.sms ? g : 4LL * sp->a.sms);
  sp->ws_common = sp->a.ws_total > sp->b.ws_total ? sp->a.ws_total : sp->b.ws_total;   // same layout, pass A's stash is the larger
  size_t o = sp->ws_common;
  sp->off_JA = o; o += (size_t)rup(n * 5 * 4, 256);
  sp->off_JB = o; o += (size_t)rup(n * 4 * 4, 256);
  sp->off_JbA = o; o += (size_t)rup(n * 5 * 4, 256);
  sp->off_JbB = o; o += (size_t)rup(n * 4 * 4, 256);
  sp->off_ps = o; o += (size_t)rup((long long)sp->blocks * 8 * 8, 256);
  sp->ws_total = o;
  return PDE_OK;
}

bool tc_supported(const pde_net* net, const pde_program* prog, long long n_points) {
  if (!program_ok(prog)) return false;
  const int order = pde_program_order(prog->kind);
  if (split_shape(net, order)) {
    SplitPlan sp;
    return make_split_plan(net, n_points, &sp) == PDE_OK;
  }
  tc::TcPlan p;
  return tc::make_plan(net, order, n_points, &p) == PDE_OK;
}

int tc_workspace_bytes(const pde_net* net, int order, long long n_points, size_t* bytes) {
  if (split_shape(net, order)) {
    SplitPlan sp;
    int rc = make_split_plan(net, n_points, &sp);
    if (rc) return rc;
    *bytes = sp.ws_total;
    return PDE_OK;
  }
  tc::TcPlan p;
  int rc = tc::make_plan(net, order, n_points, &p);
  if (rc) return rc;
  *bytes = p.ws_total;
  return PDE_OK;
}

// Shared launcher: parameter images, the fused kernel in `mode`, fixed-order reduction of the per-CTA partials.
static int tc_run(const pde_net* net, int order, int mode, const pde_envelope* env, const pde_program* prog, const void* X,
                  long long n_points, const void* seed, double inv_n, void* J, const void* Jbar, void* sums, void* grad,
                  void* energy_grad, void* workspace, size_t workspace_bytes, cudaStream_t st, const ExchangeReq* ex = nullptr) {
  using namespace tc;
  TcPlan p;
  int rc = make_plan(net, order, n_points, &p);
  if (rc) return rc;
  if ((rc = check_ptrs(net))) return rc;
  if (!X || !workspace) return PDE_ERR_INVALID;
  if (workspace_bytes < p.ws_total) return PDE_ERR_WORKSPACE;
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return PDE_ERR_INVALID;
  const TcBufs b = carve(p, workspace);
  TcArgs a = tc_args(net, p, b, X, n_points, mode, inv_n);
  a.J = static_cast<float*>(J); a.Jbar = static_cast<const float*>(Jbar);
  a.want_grad = (grad != nullptr) || (energy_grad != nullptr);
  if (mode == 0) set_program(a, env, prog, seed, inv_n);
  ReduceArgs<float> r;
  if (mode != 1 &&   // jets out: nothing to reduce
      (rc = make_reduce_args<float>(p.g, b.partial, b.psums, p.grid, 0, a.n_q, false, static_cast<float*>(grad),
                                    mode == 0 ? static_cast<float*>(sums) : nullptr,
                                    mode == 0 ? static_cast<float*>(energy_grad) : nullptr, ex, &r)))
    return rc;

  if ((rc = launch_tc_pack(net, p, b.params, b.wimg, st))) return rc;
#ifdef PDE_TC_TIMELINE
  a.dbg = timeline_buffer();
#endif
  if (launch_tc(p, a, st) != cudaSuccess) return PDE_ERR_CUDA;
  count_launch();
  set_last_path(1);
#ifdef PDE_TC_TIMELINE
  timeline_dump(a.dbg, st);
#endif
  if (mode == 1) return PDE_OK;
  if (launch_reduce<float>(st, r) != cudaSuccess) return PDE_ERR_CUDA;
  return PDE_OK;
}

// The 5-D PINN step on tensor cores: pack, forward pass A (directions 0..2) and B (3..4) writing network jets, the
// pointwise residual kernel (sums, per-point cotangents), reverse passes A and B (each recomputes its forward) whose
// reduced gradients are added, the second reduction carrying the sums, dE and, when asked for, the exchange.
static int tc_pinn_split(const pde_net* net, const pde_envelope* env, const pde_program* prog, const void* X,
                         long long n_points, const void* seed, double inv_n, void* sums, void* grad, void* energy_grad,
                         void* workspace, size_t workspace_bytes, cudaStream_t st, const ExchangeReq* ex) {
  using namespace tc;
  SplitPlan sp;
  int rc = make_split_plan(net, n_points, &sp);
  if (rc) return rc;
  if ((rc = check_ptrs(net))) return rc;
  if (!X || !workspace) return PDE_ERR_INVALID;
  if (workspace_bytes < sp.ws_total) return PDE_ERR_WORKSPACE;
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return PDE_ERR_INVALID;
  const bool want_grad = (grad != nullptr) || (energy_grad != nullptr);
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  const TcBufs b = carve(sp.a, workspace);
  float* JA = reinterpret_cast<float*>(wsb + sp.off_JA);
  float* JB = reinterpret_cast<float*>(wsb + sp.off_JB);
  float* JbA = reinterpret_cast<float*>(wsb + sp.off_JbA);
  float* JbB = reinterpret_cast<float*>(wsb + sp.off_JbB);
  double* psums_pt = reinterpret_cast<double*>(wsb + sp.off_ps);
  TcArgs pt;
  memset(&pt, 0, sizeof(pt));
  pt.X = static_cast<const float*>(X); pt.n = n_points;
  set_program(pt, env, prog, seed, inv_n);
  // With a gradient: pass A's reduction writes grad, pass B's adds to it and carries the sums, dE and the exchange.
  // Without (value or dE only): one reduction of the sums over no gradient partials.
  ReduceArgs<float> ra, rb;
  if (!grad)
    rc = make_reduce_args<float>(sp.a.g, b.partial, psums_pt, 0, sp.blocks, pt.n_q, false, nullptr,
                                 static_cast<float*>(sums), static_cast<float*>(energy_grad), ex, &rb);
  else if (!(rc = make_reduce_args<float>(sp.a.g, b.partial, psums_pt, sp.a.grid, sp.blocks, pt.n_q, false,
                                          static_cast<float*>(grad), nullptr, nullptr, nullptr, &ra)))
    rc = make_reduce_args<float>(sp.b.g, b.partial, psums_pt, sp.b.grid, sp.blocks, pt.n_q, true, static_cast<float*>(grad),
                                 static_cast<float*>(sums), static_cast<float*>(energy_grad), ex, &rb);
  if (rc) return rc;

  if ((rc = launch_tc_pack(net, sp.a, b.params, b.wimg, st))) return rc;
  auto pass = [&](const TcPlan& p, int dir0, int mode, float* J, const float* Jbar) -> int {
    TcArgs a = tc_args(net, p, b, X, n_points, mode, inv_n);
    a.dir0 = dir0; a.J = J; a.Jbar = Jbar;
    a.want_grad = mode == 2;
    if (launch_tc(p, a, st) != cudaSuccess) return PDE_ERR_CUDA;
    count_launch();
    return PDE_OK;
  };
  if ((rc = pass(sp.a, 0, 1, JA, nullptr))) return rc;
  if ((rc = pass(sp.b, 3, 1, JB, nullptr))) return rc;
  pinn_split_kernel<<<sp.blocks, SPLIT_BLOCK, 0, st>>>(pt, JA, JB, want_grad ? JbA : nullptr, want_grad ? JbB : nullptr, psums_pt);
  if (cudaGetLastError() != cudaSuccess) return PDE_ERR_CUDA;
  count_launch();
  set_last_path(1);

  if (grad) {
    if ((rc = pass(sp.a, 0, 2, nullptr, JbA))) return rc;
    if (launch_reduce<float>(st, ra) != cudaSuccess) return PDE_ERR_CUDA;
    if ((rc = pass(sp.b, 3, 2, nullptr, JbB))) return rc;
  }
  if (launch_reduce<float>(st, rb) != cudaSuccess) return PDE_ERR_CUDA;
  return PDE_OK;
}

int tc_residual_loss_grad(const pde_net* net, const pde_envelope* env, const pde_program* prog, const void* X,
                          long long n_points, const void* seed, double inv_n, void* sums, void* grad,
                          void* energy_grad, void* workspace, size_t workspace_bytes, cudaStream_t st, const ExchangeReq* ex) {
  if (!net || !prog) return PDE_ERR_INVALID;
  const int order = pde_program_order(prog->kind);
  if (order < 0) return PDE_ERR_INVALID;
  if (!program_ok(prog)) return PDE_ERR_UNSUPPORTED;
  if (split_shape(net, order)) {
    if (prog->kind != PDE_PROG_PINN) return PDE_ERR_UNSUPPORTED;
    return tc_pinn_split(net, env, prog, X, n_points, seed, inv_n, sums, grad, energy_grad, workspace, workspace_bytes, st, ex);
  }
  return tc_run(net, order, 0, env, prog, X, n_points, seed, inv_n, nullptr, nullptr, sums, grad, energy_grad, workspace,
                workspace_bytes, st, ex);
}

// Network jets on the tensor-core kernel (orders 0 and 1, whose channels are the ABI's): what the WAN losses
// evaluate for both networks at n_interior points (Poisson_ND.py:105-128, :242-276).
bool tc_jets_supported(const pde_net* net, int order, long long n_points) {
  if (order < 0 || order > 1) return false;
  tc::TcPlan p;
  return tc::make_plan(net, order, n_points, &p) == PDE_OK;
}

int tc_jets_forward(const pde_net* net, int order, const void* X, long long n_points, void* J, void* workspace,
                    size_t workspace_bytes, cudaStream_t st) {
  if (!tc_jets_supported(net, order, n_points)) return PDE_ERR_UNSUPPORTED;
  if (!J) return PDE_ERR_INVALID;
  return tc_run(net, order, 1, nullptr, nullptr, X, n_points, nullptr, 1.0, J, nullptr, nullptr, nullptr, nullptr, workspace,
                workspace_bytes, st);
}

int tc_jets_backward(const pde_net* net, int order, const void* X, long long n_points, const void* Jbar, void* grad,
                     void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (!tc_jets_supported(net, order, n_points)) return PDE_ERR_UNSUPPORTED;
  if (!Jbar || !grad) return PDE_ERR_INVALID;
  return tc_run(net, order, 2, nullptr, nullptr, X, n_points, nullptr, 1.0, nullptr, Jbar, nullptr, grad, nullptr, workspace,
                workspace_bytes, st);
}

void tc_set_path_override(int v) { tc::g_path_override.store(v < -1 || v > 1 ? -1 : v, std::memory_order_relaxed); }
int tc_get_path_override() { return tc::path_override(); }

}  // namespace pde
