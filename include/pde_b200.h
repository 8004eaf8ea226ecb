/* pde_b200.h — C ABI of the B200 collocation-point loss-step library (libpde_b200.so).
 *
 * The reference (JiakangC/Neural-Network-Based-PDE-Solver) has no FFI layer: its operator
 * boundary for this path is the set of module-level Python loss functions, which obtain
 * u, grad u, the Laplacian and the parameter gradients from nested torch.autograd calls.
 * Each entry point below names the reference interface it replaces (paths are relative to
 * the reference checkout).  INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Conventions
 *   - plain C99 types; every pointer marked "device" is CUDA device memory owned by the caller;
 *   - every call returns 0 on success or a negative pde_status; pde_strerror() names it;
 *   - nothing is allocated by the library and no state is kept between calls; all work is
 *     enqueued on `stream` (a cudaStream_t passed as void*), no host synchronisation, so the
 *     calls are CUDA-graph capturable;
 *   - floating point type is per network (PDE_F32 / PDE_F64); all device arrays of one call
 *     use that type; points X are (n, dim) row-major; jets J are (n, C) row-major with
 *     C = 1 + order*dim channels: value, dim first derivatives, dim second-derivative diagonal;
 *   - parameter gradients are written as ONE flat vector in nn.Module.parameters() order:
 *     W_0 (out,in) row-major, b_0, W_1, b_1, ...
 */
#ifndef PDE_B200_H
#define PDE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDE_ABI_VERSION 1
#define PDE_MAX_LINEAR 8   /* Linear layers per network */
#define PDE_MAX_DIM 5      /* spatial dimension d = 1..5 (README.md:23 of the reference) */
#define PDE_MAX_NODES 8    /* forced-node roots per dimension */
#define PDE_MAX_Q 4        /* per-point quantities a program may average */
#define PDE_MAX_WIDTH 256  /* hidden width */
#define PDE_MAX_PEERS 8    /* GPUs of one NVSwitch box */

typedef enum {
  PDE_OK = 0,
  PDE_ERR_INVALID = -1,      /* null pointer / bad enum / bad size */
  PDE_ERR_UNSUPPORTED = -2,  /* shape outside what the kernels implement */
  PDE_ERR_WORKSPACE = -3,    /* workspace too small */
  PDE_ERR_CUDA = -4,         /* a CUDA runtime call failed (launch, attribute) */
  PDE_ERR_NO_DEVICE = -5     /* no sm_100 device: there is no CPU fallback */
} pde_status;

enum { PDE_F32 = 0, PDE_F64 = 1 };
enum { PDE_ACT_SIN = 0, PDE_ACT_TANH = 1 };
enum { PDE_ENV_NONE = 0, PDE_ENV_POLY = 1, PDE_ENV_EXPWIN = 2 };
enum {
  PDE_PROG_PINN = 1,     /* q0 = (alpha*Lap(u) + (beta-E)*u - f)^2                order 2 */
  PDE_PROG_DRM = 2,      /* q0 = alpha*|grad u|^2 - f*u                            order 1 */
  PDE_PROG_RAYLEIGH = 3, /* q0 = alpha*|grad u|^2 + beta*u^2 ; q1 = u^2            order 1 */
  PDE_PROG_MSE = 4,      /* q0 = (u - f)^2  (f NULL -> u^2)                        order 0 */
  PDE_PROG_FLUX = 5,     /* q0 = (alpha*n.grad u + beta*u - f)^2 on box faces      order 1 */
  PDE_PROG_RITZ_VALUE = 7, /* q0 = beta*u^2/2 - g*u, g = f (f NULL -> alpha)       order 0 */
  PDE_PROG_PARABOLIC = 9   /* q0 = (du/dt + alpha*Lap_x(u) + (beta-E)*u - f)^2, t = x_{dim-1}  order 2 */
};
/* Kinds 6 and 8 are not assigned: the library has always answered PDE_ERR_INVALID for them, and stays so for callers
 * that check that answer. */

/* Faces of the box [lo, hi]^dim for PDE_PROG_FLUX and pde_sample_faces_rhs: face k is x_{k/2} = lo (outward normal
 * -e_{k/2}) when k is even and x_{k/2} = hi (normal +e_{k/2}) when k is odd.  A face set is a bit mask over bits
 * 0 .. 2*dim-1.  A batch of n face points is popcount(mask) equal contiguous blocks, one per set bit in increasing bit
 * order: point p lies on the face of set bit number p / (n / popcount(mask)).  The kernels need only the axis and the
 * sign of the normal, never lo or hi.  With every face set (mask (1 << 2*dim) - 1) a pure-Neumann problem is
 * accepted; its solution is determined only up to a constant. */

/* A fully connected network [dim, H, ..., H, 1] with sin or tanh activations.
 * Replaces: SolutionNet / CriticNet (Poisson_Equations/Poisson_ND.py:11-46), FCN
 * (Schrodinger_Equations/.../IPW_1D_WAN.py:62-81, QHO_2D.py:103-114), FCN1D (KH_1D.py:104-112).
 * W[l] is nn.Linear.weight of layer l, (widths[l+1], widths[l]) row-major; b[l] its bias. */
typedef struct pde_net {
  int32_t dtype;                      /* PDE_F32 | PDE_F64 */
  int32_t dim;                        /* 1..PDE_MAX_DIM */
  int32_t n_linear;                   /* 2..PDE_MAX_LINEAR */
  int32_t activation;                 /* PDE_ACT_* */
  int32_t widths[PDE_MAX_LINEAR + 1]; /* widths[0]=dim, hidden widths equal, widths[n_linear]=1 */
  const void* W[PDE_MAX_LINEAR];      /* device */
  const void* b[PDE_MAX_LINEAR];      /* device */
} pde_net;

/* Separable hard-constraint envelope u = B(x) * net(x), B = prod_i b(x_i).
 * PDE_ENV_POLY   b(t) = (t-lo)(hi-t)                      Poisson_ND.py:27-29, IPW_1D_WAN.py:77-80
 * PDE_ENV_EXPWIN b(t) = (1-exp(-(t-lo)))(1-exp(t-hi))     QHO_2D.py:149-153, KH_1D.py:117-120
 * nodes: b(t) additionally times prod_k (t - nodes[i][k])  IPW_1D_PINN_DRM.py:44-51, QHO_2D.py:155-168 */
typedef struct pde_envelope {
  int32_t kind;
  int32_t n_nodes[PDE_MAX_DIM];
  double lo, hi;
  double nodes[PDE_MAX_DIM][PDE_MAX_NODES];
} pde_envelope;

/* Per-point residual program evaluated on the jets of u = B*net.
 * f, beta: optional device arrays of n values; energy: optional device scalar (trainable E,
 * KH_1D.py:218, QHO_2D_Energy.py:287-291), else energy_const.
 * PDE_PROG_FLUX is the boundary-flux penalty of a Neumann (beta = 0) or Robin condition: f holds the prescribed data g
 * (NULL: g = 0), beta (or beta_const) the Robin coefficient, `faces` the face mask of the points (layout above); the
 * energy fields are ignored and dq/dE = 0.  The reference has no Neumann code (its README.md:23 advertises it).
 * PDE_PROG_RITZ_VALUE is the value-only term of a Deep Ritz functional (DESIGN.md §3.4b): q0 = beta*u^2/2 - g*u with
 * beta from `beta` (or beta_const) and g from f, or the constant alpha when f is NULL; `faces` and the energy fields
 * are ignored and dq/dE = 0.  It needs no normal, so the points may lie on any boundary.  Its uses: the Robin /
 * Neumann boundary energy (beta = kappa, f = g on boundary points; the reference has no counterpart, its
 * drm_energy_loss, Poisson_ND.py:98-103, is the interior half of the same functional) and the integral of u for a
 * mean constraint (beta = 0, f = NULL, alpha = -1: q0 = u, with the caller's seed).
 * PDE_PROG_PARABOLIC is the space-time residual of a parabolic equation (DESIGN.md §3.4c).  The LAST coordinate is time:
 * x = (x_0 .. x_{dim-2}, t), dim = 2..5, and Lap_x = sum_{i < dim-1} d^2/dx_i^2 is the spatial Laplacian.  beta, E and
 * f are as for PDE_PROG_PINN (per-point or constant beta, energy pointer or constant, f NULL -> 0), dq/dE = -2 r u.  The
 * heat equation u_t = kappa Lap_x u + s is alpha = -kappa, beta = 0, f = s.  In the face layout above the spatial faces
 * are the mask (1 << 2*(dim-1)) - 1 and the initial face t = lo is bit 2*(dim-1): initial and boundary data are
 * PDE_PROG_MSE (or PDE_PROG_FLUX) calls on such points.  The program uses the jets of order 2, so
 * pde_workspace_bytes(net, 2, n) covers it on both kernel families, and it has as many jet channels as PDE_PROG_PINN at
 * the same dim. */
typedef struct pde_program {
  int32_t kind;        /* PDE_PROG_* */
  int32_t faces;       /* PDE_PROG_FLUX: face mask, 1 .. (1 << 2*dim) - 1; ignored by every other program */
  double alpha;
  double beta_const;   /* used when beta == NULL */
  double energy_const; /* used when energy == NULL */
  const void* f;       /* device, (n) or NULL */
  const void* beta;    /* device, (n) or NULL */
  const void* energy;  /* device scalar or NULL */
} pde_program;

int pde_abi_version(void);
const char* pde_strerror(int status);

/* Number of parameters (length of the flat gradient vector). */
int pde_param_count(const pde_net* net, int64_t* n_params);

/* Jet channels for (dim, order) and number of averaged quantities of a program kind. */
int pde_jet_channels(int32_t dim, int32_t order);
int pde_program_quantities(int32_t kind);
int pde_program_order(int32_t kind);

/* Workspace bytes needed by any of the calls below for this network / order / n points. */
int pde_workspace_bytes(const pde_net* net, int32_t order, int64_t n_points, size_t* bytes);

/* Network jets (value, gradient, Hessian diagonal of net(X), no envelope).
 * Replaces: model.net(X) + grad_scalar_field + laplacian (Poisson_ND.py:61-71),
 * compute_derivatives (QHO_1D_PINN_DRM.py:155-160).  J: device (n, C). */
int pde_jets_forward(const pde_net* net, int32_t order, const void* X, int64_t n_points,
                     void* J, void* workspace, size_t workspace_bytes, void* stream);

/* Reverse sweep of pde_jets_forward: grad[k] = sum_p sum_c Jbar[p,c] dJ[p,c]/dtheta_k.
 * Replaces: loss.backward() through the nested autograd graph (Poisson_ND.py:240).
 * The forward is recomputed tile by tile on chip; nothing but X and Jbar is read. */
int pde_jets_backward(const pde_net* net, int32_t order, const void* X, int64_t n_points,
                      const void* Jbar, void* grad, void* workspace, size_t workspace_bytes,
                      void* stream);

/* Fused loss step: forward jets, envelope, residual program, per-point seeds and the reverse
 * sweep in one pass per tile of points.
 * Replaces: pinn_residual_loss / drm_energy_loss (+ .backward()) (Poisson_ND.py:91-103,:240),
 * PINN_loss / DRM_loss (IPW_1D_PINN_DRM.py:63-90), pinn_loss / drm_loss (KH_1D.py:226-242),
 * the inline residual blocks (QHO_2D.py:363-383, IPW_2D.py:195-228), boundary / data / norm
 * value terms (Poisson_ND.py:130-147,230-232).
 *   sums   : device (K) out — sum_p q_k(p) (raw sums; the caller divides by its global N)
 *   grad   : device (n_params) out or NULL — sum_k seed[k] * inv_n * sum_p dq_k(p)/dtheta
 *   energy_grad : device scalar out or NULL — same contraction for dq/dE
 *   seed   : device (K) or NULL (all ones) — dLoss/dmean_k, lets functions of means
 *            (Rayleigh quotient, WAN) and multi-GPU exact recombination share one kernel.
 * A PDE_PROG_FLUX call returns PDE_ERR_INVALID, before it enqueues anything, when faces == 0,
 * faces >= 1 << 2*dim or n_points is not a multiple of popcount(faces); so does the _exchange variant below.
 * A PDE_PROG_PARABOLIC call returns PDE_ERR_INVALID, before it enqueues anything, when dim < 2 (there is no spatial
 * axis) or when env is non-NULL with a kind other than PDE_ENV_NONE or any n_nodes[i] != 0: every envelope vanishes at
 * both ends of every axis, the time axis included, which is wrong for an initial-value problem.  So does the _exchange
 * variant below. */
int pde_residual_loss_grad(const pde_net* net, const pde_envelope* env, const pde_program* prog,
                           const void* X, int64_t n_points, const void* seed, double inv_n,
                           void* sums, void* grad, void* energy_grad, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Which kernel family pde_residual_loss_grad uses for this network / program / size:
 * 0 = generic SIMT FMA kernel, 1 = tcgen05 tensor-core kernel; negative = pde_status. Pure query. */
int pde_query_path(const pde_net* net, const pde_program* prog, int64_t n_points);

/* Same query for pde_jets_forward / pde_jets_backward (orders 0 and 1 run on the tcgen05 kernel for fp32 networks
 * [d, H<=64, ...] above 4096 points, e.g. both networks of wan_losses at n_interior points, Poisson_ND.py:105-128). */
int pde_query_jets_path(const pde_net* net, int32_t order, int64_t n_points);

/* Kernel-family override, process wide: -1 automatic (default; initial value from PDE_B200_PATH=simt|tc, read once),
 * 0 generic SIMT kernel always, 1 tcgen05 kernel for every shape it implements regardless of the point count.
 * The parity tests use it to run both families on identical inputs.  There is no reference counterpart. */
int pde_set_kernel_path(int32_t path);
int pde_kernel_path(void);

/* Which family the calling thread's last fused / jets call actually launched (0 SIMT, 1 tcgen05, -1 none yet), and
 * how many kernels this library has enqueued in the process so far (every launch site counts itself).  Host-side
 * bookkeeping for bench.py's `kernel_path` and `gpu_launches` fields; no reference counterpart. */
int pde_last_kernel_path(void);
uint64_t pde_launch_count(void);

/* WAN weak-form coupling of two networks on their jets (order 1), elementwise.
 * Replaces: bump_w + wan_losses (Poisson_ND.py:74-88,105-128), function_w + WAN_loss
 * (IPW_1D_WAN.py:31-59,88-115; QHO_2D.py:172-225), weight_fn_w + wan_loss (KH_1D.py:138-148,244-269).
 *   q0 = alpha*grad u . grad phi + (beta-E)*u*phi - f*phi, q1 = phi^2, q2 = u^2, q3 = |grad v|^2 + v^2,
 *   phi = w*v, w = prod_i bump((x_i-c)/h) on [w_lo, w_hi], bump(t) = exp(1/(t^2-1+eps_den))/0.210987.
 *   Ju, Jv  : device (n, 1+dim) network jets of u-net / v-net (pde_jets_forward, order 1)
 *   sums    : device (5) out — sum_p q0..q3 and sum_p dq0/dE
 *   seed    : device (4) or NULL; when Jbar_u / Jbar_v are non-NULL they receive
 *             sum_k seed[k]*inv_n*dq_k/dJ (cotangents for pde_jets_backward). */
typedef struct pde_wan {
  int32_t dtype, dim;
  double alpha, beta_const, energy_const, w_lo, w_hi, eps_den;
  const void* f;      /* device (n) or NULL */
  const void* beta;   /* device (n) or NULL */
  const void* energy; /* device scalar or NULL */
  pde_envelope env_u, env_v;
} pde_wan;

int pde_wan_pointwise(const pde_wan* wan, const void* X, int64_t n_points, const void* Ju,
                      const void* Jv, const void* seed, double inv_n, void* sums, void* Jbar_u,
                      void* Jbar_v, void* workspace, size_t workspace_bytes, void* stream);

/* The scalar end of the WAN losses in one launch: out = (loss_pde, loss_v, loss_norm, total) of the four means of
 * pde_wan_pointwise and jac = d out_i / d mean_j (4 x 4, row major), both device arrays of the given dtype.
 *   kind 0: loss_pde = m0^2 / (m1 + eps_pde)                          Poisson_ND.py:118-122, IPW_1D_WAN.py:108-110, QHO_2D.py:218-219
 *   kind 1: loss_pde = (vol m0 / (vol m1 + eps_pde))^2               KH_1D.py:263-267
 *   loss_v = -log(loss_pde + eps_log) + reg m3;  loss_norm = (vol m2 - 1)^2;  total = w_pde loss_pde + w_norm loss_norm
 *   consts (host, 6 doubles): eps_pde, eps_log, vol, reg, w_pde, w_norm.
 * Replaces: the ~25 zero-dimensional tensor operations (and their autograd nodes) each reference WAN_loss ends with. */
int pde_wan_scalars(int32_t dtype, int32_t kind, const void* means, const double* consts, void* out, void* jac,
                    void* stream);

/* ---- the device-side pieces of an epoch around the loss step (all single launches, graph capturable) ---- */

/* Collocation-point sampling with the manufactured solution / right-hand side in the same pass.
 * Replaces: sample_interior (Poisson_ND.py:187-190: X = rand(N, d) * L), exact_u_prod_sin and
 * rhs_f_for_u_sin (Poisson_ND.py:49-58), and the test-point draw of the L2 evaluation (:281-285).
 *   X (n, dim) out: lo + (hi-lo) * U[0,1), Philox4x32-10 keyed by `seed`, counter = (point index, `offset`
 *                   + *offset_add when that optional device int64 is given, e.g. the Adam step counter, so
 *                   that a replayed CUDA graph draws fresh points every epoch);
 *                   statistically equivalent to torch.rand, not bit-identical (SURVEY.md §8f-1).
 *   X_in: when non-NULL the points are read from X_in instead of sampled (X may be NULL).
 *   k (host, dim) and period: u_exact = prod_i sin(k_i pi x_i / period), f = sum_i (k_i pi / period)^2 u_exact;
 *   u_exact, f: device (n) out, each optional. */
int pde_sample_points_rhs(int32_t dtype, int32_t dim, int64_t n_points, double lo, double hi, uint64_t seed,
                          uint64_t offset, const void* offset_add, const double* k, double period,
                          const void* X_in, void* X, void* u_exact, void* f, void* stream);

/* Face points with the manufactured Neumann data in the same pass.
 * Replaces: the face draw of boundary_loss_dirichlet (Poisson_ND.py:130-141: X = rand(N, d) * L, X[:, i] = 0 or L),
 * extended to a face mask (layout at pde_program above) and to the outward normal derivative of the manufactured
 * solution of Poisson_ND.py:49-58.
 *   X (popcount(faces) * n_per_face, dim) out: point p has exactly the coordinates pde_sample_points_rhs draws for
 *     point index p with the same seed, offset and offset_add (same Philox counter, same half-open clamp), then the
 *     face coordinate of its block set to lo or hi;
 *   g: device (n) out or NULL (needs k and period): g = s (k_a pi / P) cos(k_a pi x_a / P) prod_{j != a} sin(k_j pi x_j / P),
 *     s = -1 on the lo face and +1 on the hi face of axis a. */
int pde_sample_faces_rhs(int32_t dtype, int32_t dim, int64_t n_per_face, int32_t faces, double lo, double hi,
                         uint64_t seed, uint64_t offset, const void* offset_add, const double* k, double period, void* X,
                         void* g, void* stream);

/* Fused Adam over the flat gradient vector that pde_residual_loss_grad writes (parameters() order, a
 * trailing trainable energy scalar included when it is listed as the last tensor).
 * Replaces: torch.optim.Adam(model.parameters(), lr).step() (Poisson_ND.py:177,240; KH_1D.py:330-336).
 *   m += (1-beta1)(g-m);  v = beta2 v + (1-beta2) g^2;  p -= lr/(1-beta1^t) * m / (sqrt(v)/sqrt(1-beta2^t) + eps)
 *   with g = grad_scale * grad_flat[i] (+ weight_decay * p), t = *step + 1; *step is incremented (device int64). */
typedef struct pde_adam {
  int32_t dtype;
  int32_t n_tensors;                      /* 1 .. 2*PDE_MAX_LINEAR+1 */
  double lr, beta1, beta2, eps, weight_decay, grad_scale;
  void* param[2 * PDE_MAX_LINEAR + 1];    /* device: the nn.Parameter storages, updated in place */
  int64_t numel[2 * PDE_MAX_LINEAR + 1];
} pde_adam;

int pde_adam_step(const pde_adam* cfg, const void* grad_flat, void* exp_avg, void* exp_avg_sq, void* step,
                  void* stream);

/* Device-side best-model tracking: if *metric < *best_metric, copy every parameter tensor into best_flat
 * and update *best_metric (and *best_step = *step when both are given).  No host read-back.
 * Replaces: the per-epoch `.item()` + state_dict copy to the CPU (Poisson_ND.py:288-300). */
int pde_keep_best(const pde_adam* cfg, const void* metric, void* best_metric, void* best_flat, const void* step,
                  void* best_step, void* stream);

/* ---- exchange step of the data-parallel loss step over NVLink peer memory (one kernel, no NCCL call) ---- */

/* Peer-visible buffers: plain device allocations shared through CUDA IPC handles (64 bytes, exchanged by
 * the host side once at set-up).  pde_peer_bytes gives the size for a given slot capacity:
 * [control words | parity 0: per source rank (value, flag) pairs | parity 1]. */
int pde_peer_bytes(int32_t dtype, int64_t slot_elems, size_t* bytes);
int pde_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);   /* cudaMalloc + zero + cudaIpcGetMemHandle */
int pde_peer_open(const unsigned char* handle64, void** ptr);            /* cudaIpcOpenMemHandle (another process' buffer) */
int pde_peer_close(void* ptr);
int pde_peer_free(void* ptr);

typedef struct pde_peers {
  int32_t rank, world;             /* world <= PDE_MAX_PEERS */
  void* base[PDE_MAX_PEERS];       /* base[r]: rank r's buffer as mapped in THIS process (own allocation at base[rank]) */
} pde_peers;

/* In-place sum of `buf` (n values) over the ranks of one box, flag-in-data push protocol: every 32-bit word
 * is stored together with the call number as one 64-bit word into every peer's slot (one one-way NVLink trip,
 * no fence, no separate signal); the rank then polls its own slots and adds the values in rank order
 * (bit-identical result on every rank, independent of arrival order).  One launch; `seq` (device uint32,
 * zero at start) counts the calls so the kernel can be replayed from a CUDA graph.  A peer that does not
 * arrive within the exchange timeout (below) poisons the result with NaN instead of hanging the GPU.
 * Replaces: the gradient exchange a data-parallel run of train_poisson_nd needs after loss.backward()
 * (Poisson_ND.py:240; the reference itself is single-device), SURVEY.md §8e. */
int pde_allreduce_oneshot(const pde_peers* peers, int32_t dtype, void* buf, int64_t n, int64_t slot_elems,
                          void* seq, void* stream);

/* The fused loss step with the exchange folded into its reduction (SURVEY.md §8f-4): the kernel that sums the per-CTA
 * partial gradients pushes every reduced element to the peers, collects theirs and writes the rank-ordered sum, so a
 * data-parallel step is pack + fused kernel + reduce-and-exchange — no separate all-reduce launch.
 *   result : device, [grad (n_params) | dE (1) | sums (K)] contiguous, every element summed over the ranks
 *   peers, slot_elems (>= n_params + 1 + K), seq : as for pde_allreduce_oneshot (same buffers, same call counter).
 * Replaces: loss.backward() + the gradient exchange of a data-parallel train_poisson_nd step (Poisson_ND.py:240). */
int pde_residual_loss_grad_exchange(const pde_net* net, const pde_envelope* env, const pde_program* prog,
                                    const void* X, int64_t n_points, const void* seed, double inv_n, void* result,
                                    void* workspace, size_t workspace_bytes, const pde_peers* peers,
                                    int64_t slot_elems, void* seq, void* stream);

/* Failure reporting of the exchange.  Every rank must make the same sequence of pde_allreduce_oneshot calls
 * (lockstep, as for any collective).  A rank waits for its peers for at most the exchange timeout — process wide,
 * default 600 s, 0 = for ever — and on expiry poisons ITS OWN result with NaN and counts the event in its control
 * block; peers that did receive this rank's words are not affected and cannot know, so the host must look:
 * pde_exchange_errors synchronises `stream` and returns the number of timed-out elements seen so far on this rank. */
int pde_set_exchange_timeout(double seconds);
int pde_exchange_errors(const pde_peers* peers, uint32_t* timeouts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PDE_B200_H */
