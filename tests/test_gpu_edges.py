"""GPU parity tests of the C ABI at the edges of its advertised envelope (run with -m gpu on a B200).

include/pde_b200.h promises dim 1..5, 2..8 Linear layers, hidden widths 1..256, up to PDE_MAX_NODES forced nodes per
dimension, a trainable-energy pointer with its gradient, a free seed vector and inv_n, and any n >= 1.  The reference
shapes the other parity tests use stay well inside that envelope; here the ABI is driven directly through the ctypes
structs, every output buffer and the workspace belong to the test (so they can be poisoned), and the reference is the
float64 numpy oracle (oracle/jets_numpy).  The cases sit where kernels go wrong: one hidden layer, width 1 (padded to 8
units) and 256 (two warps per point, W streamed in K-chunks), the deepest net, tile tails, tensor-core options that the
reference shapes never reach, and the decline edges between the two kernel families.  Every program of the header runs
here: PINN, DRM, RAYLEIGH and MSE, the boundary flux (FLUX, on the blocked face layout), the Ritz value term (RITZ) and
the space-time parabolic residual (PARABOLIC), the last three also with the fields the header says they ignore (g).

Bars: 1e-10 in fp64 and 1e-5 in fp32 (conftest.BASE_TOL), on the sums, on every parameter gradient
(conftest.assert_grads_close) and on dE.  Inputs of fp32 cases are fp32-representable, so the oracle sees exactly
what the kernel sees."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from conftest import BASE_TOL, assert_grads_close
from oracle import jets_numpy as O

pytestmark = pytest.mark.gpu

PAD = 16            # elements past the end of every output buffer; a call must leave them as they were
POISON = 0xFF       # all-ones bytes: NaN in fp32 and fp64
PINN, DRM, RAYLEIGH, MSE, FLUX, RITZ, PARABOLIC = 1, 2, 3, 4, 5, 7, 9
ORDER = {PINN: 2, DRM: 1, RAYLEIGH: 1, MSE: 0, FLUX: 1, RITZ: 0, PARABOLIC: 2}
NQ = {PINN: 1, DRM: 1, RAYLEIGH: 2, MSE: 1, FLUX: 1, RITZ: 1, PARABOLIC: 1}
NAME = {PINN: "pinn", DRM: "drm", RAYLEIGH: "ray", MSE: "mse", FLUX: "flux", RITZ: "ritz", PARABOLIC: "par"}
SIN, TANH = O.SIN, O.TANH
F32, F64 = torch.float32, torch.float64


def _lib():
    from pde_b200 import _lib as L
    return L, L.load()


def _path(which):
    import pde_b200 as pb
    return pb.ops.kernel_path(which)


def _tol(dtype):
    return BASE_TOL[str(dtype).replace("torch.", "")]


def _rnd(a, dtype):
    """What the kernel of `dtype` sees of a float64 array (fp32 cases round every input once)."""
    a = np.asarray(a, dtype=np.float64)
    return a.astype(np.float32).astype(np.float64) if dtype == F32 else a


def _rand_net(rng, d, w, n_linear, dtype):
    """tests/test_gpu_tc._rand_net: fan-in-scaled uniform weights, fp32-representable values."""
    Ws = [rng.uniform(-1, 1, (w, d)) / math.sqrt(d)] + [rng.uniform(-1, 1, (w, w)) / math.sqrt(w)
                                                        for _ in range(n_linear - 2)] + [rng.uniform(-1, 1, (1, w)) / math.sqrt(w)]
    bs = [rng.uniform(-0.5, 0.5, W.shape[0]) for W in Ws]
    return [_rnd(_rnd(W, F32), dtype) for W in Ws], [_rnd(_rnd(b, F32), dtype) for b in bs]


def _dev(a, dtype):
    return torch.tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class _Net:
    """A pde_net over device copies of (Ws, bs)."""

    def __init__(self, Ws, bs, act, dtype):
        L, _ = _lib()
        self.Ws, self.bs, self.act, self.dtype = Ws, bs, act, dtype
        self.t = [(_dev(W, dtype), _dev(b, dtype)) for W, b in zip(Ws, bs)]
        c = L.Net()
        c.dtype = L.F64 if dtype == F64 else L.F32
        c.dim, c.n_linear, c.activation = Ws[0].shape[1], len(Ws), act
        c.widths[0] = c.dim
        for l, (W, b) in enumerate(self.t):
            c.widths[l + 1] = W.shape[0]
            c.W[l], c.b[l] = W.data_ptr(), b.data_ptr()
        self.c = c
        self.n_params = sum(W.size + b.size for W, b in zip(Ws, bs))

    def unflat(self, g):
        g = g.double().cpu().numpy()
        gWs, gbs, o = [], [], 0
        for W, b in zip(self.Ws, self.bs):
            gWs.append(g[o:o + W.size].reshape(W.shape)); o += W.size
            gbs.append(g[o:o + b.size]); o += b.size
        assert o == g.size
        return gWs, gbs


def _envelope(kind, lo=0.0, hi=2.0, nodes=(), dtype=F64):
    """(pde_envelope, oracle envelope dict) of one description; node positions rounded as the kernel sees them."""
    L, _ = _lib()
    nodes = [list(_rnd(ns, dtype)) for ns in nodes]
    e = L.Envelope()
    e.kind, e.lo, e.hi = kind, lo, hi
    for i, ns in enumerate(nodes):
        e.n_nodes[i] = len(ns)
        for k, v in enumerate(ns):
            e.nodes[i][k] = v
    return e, {"kind": kind, "lo": lo, "hi": hi, "nodes": nodes or None}


def _cheb(k, lo=-2.0, hi=2.0):
    """k Chebyshev points of [lo, hi]: the product of (x - node) stays within 2 ((hi - lo) / 4)^k on the interval."""
    return [0.5 * (lo + hi) + 0.5 * (hi - lo) * math.cos((2 * j + 1) * math.pi / (2 * k)) for j in range(k)]


def _buf(n, dtype, fill):
    """n elements followed by PAD sentinel elements, every byte = fill."""
    es = torch.tensor([], dtype=dtype).element_size()
    return torch.full(((n + PAD) * es,), fill, dtype=torch.uint8, device="cuda").view(dtype)


def _untouched_tail(buf, n, fill):
    es = buf.element_size()
    return bool((buf.view(torch.uint8)[n * es:] == fill).all())


def _bytes(t, n):
    return t.view(torch.uint8)[:n * t.element_size()].cpu()


def _workspace(net, order, n, fill):
    L, lib = _lib()
    nb = C.c_size_t(0)
    L.check(lib.pde_workspace_bytes(C.byref(net.c), order, n, C.byref(nb)), "pde_workspace_bytes")
    return torch.full((max(nb.value, 256),), fill, dtype=torch.uint8, device="cuda")


class _Case:
    """Points, per-point arrays and program of one pde_residual_loss_grad call (float64 host copies + device copies)."""

    def __init__(self, net, env, kind, X, alpha=1.0, f=None, beta=None, beta_const=0.0, E=0.0, energy_ptr=False, faces=0):
        L, _ = _lib()
        dt = net.dtype
        self.net, self.env_c, self.env = net, env[0], env[1]
        self.kind, self.alpha, self.faces = kind, alpha, faces
        self.X = _rnd(X, dt)
        self.n = self.X.shape[0]
        self.f = None if f is None else _rnd(np.asarray(f).reshape(-1, 1), dt)
        self.beta = None if beta is None else _rnd(np.asarray(beta).reshape(-1, 1), dt)
        self.beta_const, self.E = float(_rnd(beta_const, dt)), float(_rnd(E, dt))
        self.Xd = _dev(self.X, dt)
        self.fd = None if f is None else _dev(self.f.reshape(-1), dt)
        self.bd = None if beta is None else _dev(self.beta.reshape(-1), dt)
        self.Ed = _dev(np.array([self.E]), dt) if energy_ptr else None
        p = L.Program()
        p.kind, p.faces, p.alpha, p.beta_const = kind, faces, alpha, self.beta_const
        p.energy_const = 0.0 if energy_ptr else self.E      # with the pointer the constant must not be read
        p.f, p.beta, p.energy = _ptr(self.fd), _ptr(self.bd), _ptr(self.Ed)
        self.prog = p

    def run(self, seed=None, inv_n=None, fill=0, grad=True, dE=True, sums=True, ws=None):
        """One pde_residual_loss_grad call on buffers this test owns (filled with `fill`). Returns the outputs (first
        K / n_params / 1 elements), the kernel family that served the call and whether every sentinel survived."""
        L, lib = _lib()
        dt, K = self.net.dtype, NQ[self.kind]
        ws = _workspace(self.net, ORDER[self.kind], self.n, fill) if ws is None else ws
        out = {"sums": _buf(K, dt, fill) if sums else None, "grad": _buf(self.net.n_params, dt, fill) if grad else None,
               "dE": _buf(1, dt, fill) if dE else None}
        sd = None if seed is None else _dev(_rnd(seed, dt), dt)
        rc = lib.pde_residual_loss_grad(C.byref(self.net.c), C.byref(self.env_c), C.byref(self.prog), self.Xd.data_ptr(),
                                        self.n, _ptr(sd), 1.0 / self.n if inv_n is None else inv_n, _ptr(out["sums"]),
                                        _ptr(out["grad"]), _ptr(out["dE"]), ws.data_ptr(), ws.numel(), _stream())
        L.check(rc, "pde_residual_loss_grad")
        torch.cuda.synchronize()
        lens = {"sums": K, "grad": self.net.n_params, "dE": 1}
        intact = all(_untouched_tail(b, lens[k], fill) for k, b in out.items() if b is not None)
        res = {k: (None if b is None else b[:lens[k]]) for k, b in out.items()}
        res["path"], res["intact"], res["ws"] = lib.pde_last_kernel_path(), intact, ws
        return res

    def query_path(self):
        _, lib = _lib()
        return lib.pde_query_path(C.byref(self.net.c), C.byref(self.prog), self.n)

    def oracle(self, seed=None, inv_n=None):
        """sums_k = sum_p q_k, grad = sum_k seed_k inv_n sum_p dq_k/dtheta, dE = seed_0 inv_n sum_p dq_0/dE, restated on
        oracle/jets_numpy (the programs of include/pde_b200.h), with the scales the comparisons use: sum_p |q_k| and
        seed_0 inv_n sum_p |dq_0/dE|."""
        net, d, kind, a = self.net, self.X.shape[1], self.kind, self.alpha
        K = NQ[kind]
        w = (np.ones(K) if seed is None else _rnd(seed, net.dtype)) * (1.0 / self.n if inv_n is None else inv_n)
        beta = self.beta if self.beta is not None else self.beta_const
        f = 0.0 if self.f is None else self.f

        def program(U):
            u, g = U[:, 0:1], U[:, 1:1 + d]
            Ub = np.zeros_like(U)
            dE = dEs = 0.0
            if kind == PINN:
                q, Ub, _ = O.pinn_program(U, d, self.f, alpha=a, beta=beta, E=self.E)
                r = a * np.sum(U[:, 1 + d:1 + 2 * d], axis=1, keepdims=True) + (beta - self.E) * u - f
                qs, Ub = [q], w[0] * Ub
                dE, dEs = w[0] * float(np.sum(-2.0 * r * u)), abs(w[0]) * float(np.sum(np.abs(2.0 * r * u)))
            elif kind == DRM:
                qs = [a * np.sum(g * g, axis=1, keepdims=True) - f * u]
                Ub[:, 0:1] = -w[0] * f
                Ub[:, 1:1 + d] = w[0] * 2.0 * a * g
            elif kind == RAYLEIGH:
                (q1, q2), (U1, U2) = O.rayleigh_program(U, d, a, beta)
                qs, Ub = [q1, q2], w[0] * U1 + w[1] * U2
            elif kind == FLUX:      # no dq/dE: dE must come back as exactly 0
                q, U0 = O.flux_program(U, d, self.faces, self.f, a, beta)
                qs, Ub = [q], w[0] * U0
            elif kind == RITZ:
                q, U0 = O.ritz_value_program(U, self.f, a, beta)
                qs, Ub = [q], w[0] * U0
            elif kind == PARABOLIC:
                q, U0, dE0 = O.parabolic_program(U, d, self.f, alpha=a, beta=beta, E=self.E)
                qs, Ub = [q], w[0] * U0
                dE, dEs = w[0] * dE0, abs(w[0]) * float(np.sum(np.abs(U0[:, d:d + 1] * u)))   # U0[:, d] = 2 r
            else:
                r = u - f
                qs = [r * r]
                Ub[:, 0:1] = w[0] * 2.0 * r
            return [float(np.sum(q)) for q in qs], Ub, ([float(np.sum(np.abs(q))) for q in qs], dE, dEs)

        sums, gWs, gbs, (scales, dE, dEs) = O._loss_and_grads(net.Ws, net.bs, self.X, net.act, ORDER[kind], self.env, program)
        return {"sums": np.array(sums), "sum_scales": np.array(scales), "grads": (gWs, gbs), "dE": dE, "dE_scale": dEs}


def _assert_matches_oracle(case, got, want, what, dE=True):
    tol = _tol(case.net.dtype)
    s = got["sums"].double().cpu().numpy()
    for k in range(len(s)):
        e = abs(s[k] - want["sums"][k]) / max(want["sum_scales"][k], 1e-300)
        assert e <= tol, f"{what}: sum {k} {s[k]!r} vs {want['sums'][k]!r}: {e:.3e} > {tol:.1e}"
    assert_grads_close(case.net.unflat(got["grad"]), want["grads"], tol, what)
    if dE and got["dE"] is not None:
        g = float(got["dE"][0])
        e = abs(g - want["dE"]) / max(want["dE_scale"], 1e-300)
        assert e <= tol, f"{what}: dE {g!r} vs {want['dE']!r}: {e:.3e} > {tol:.1e}"
    assert got["intact"], f"{what}: an output was written past its end"


def _points(rng, n, d, lo=0.05, hi=1.95):
    return rng.uniform(lo, hi, (n, d))


# ================================================================================================ (a) planner coverage
HS = (1, 2, 3, 4, 5, 8, 63, 64, 65, 127, 128, 200, 255, 256)


def test_planner_covers_the_advertised_envelope():
    """pde_workspace_bytes plans, and pde_query_path names a kernel family for, every shape include/pde_b200.h admits:
    both dtypes, dim 1..5, order 0..2, 2..8 Linear layers, widths from 1 to 256 around every padding and chunk edge —
    at one point and at 8192, with the kernel family chosen automatically and forced onto the tensor cores.  Every
    program of each order is asked: MSE and RITZ (order 0), DRM and FLUX on all 2d faces (order 1), PINN and, from
    d = 2, PARABOLIC (order 2).  The tensor-core kernel has no 5-D parabolic pass, so there PARABOLIC answers 0."""
    L, lib = _lib()
    progs = {0: (MSE, RITZ), 1: (DRM, FLUX), 2: (PINN, PARABOLIC)}
    refused = []
    for which in ("auto", "tc"):
        with _path(which):
            for dt in (L.F32, L.F64):
                for d in range(1, 6):
                    for order in range(3):
                        for kind in progs[order]:
                            if kind == PARABOLIC and d == 1:
                                continue
                            prog = L.Program()
                            prog.kind = kind
                            prog.faces = (1 << 2 * d) - 1 if kind == FLUX else 0
                            for nl in range(2, 9):
                                for H in HS:
                                    net = L.Net()
                                    net.dtype, net.dim, net.n_linear, net.activation = dt, d, nl, L.ACT_SIN
                                    net.widths[0] = d
                                    for l in range(1, nl):
                                        net.widths[l] = H
                                    net.widths[nl] = 1
                                    for n in (1, 8192):
                                        nb = C.c_size_t(0)
                                        rc = lib.pde_workspace_bytes(C.byref(net), order, n, C.byref(nb))
                                        path = lib.pde_query_path(C.byref(net), C.byref(prog), n)
                                        ok = (0,) if kind == PARABOLIC and d == 5 else (0, 1)
                                        if rc != 0 or nb.value == 0 or path not in ok:
                                            refused.append(("f64" if dt == L.F64 else "f32", f"d={d}", NAME[kind],
                                                            f"n_linear={nl}", f"H={H}", f"n={n}", which, rc, path))
    assert not refused, f"{len(refused)} shapes inside the header's envelope refused: {refused}"


# ================================================================================================ (b) generic kernel
# dtype, d, n_linear, H, activation, program, envelope (kind, lo, hi, nodes), N, energy through the pointer
ENV_POLY02 = (O.ENV_POLY, 0.0, 2.0, ())
ENV_NONE02 = (O.ENV_NONE, 0.0, 2.0, ())
GENERIC = [
    (F64, 5, 8, 256, SIN, PINN, ENV_POLY02, 7, True),          # the widest, deepest fp64 order-2 net: KC below default
    (F64, 5, 8, 255, TANH, RAYLEIGH, ENV_POLY02, 2, False),
    (F64, 1, 8, 256, TANH, PINN, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(3),)), 149, False),
    (F64, 5, 2, 1, SIN, PINN, ENV_POLY02, 1000, True),         # one hidden layer (n_h == 1) of one unit
    (F64, 1, 2, 3, TANH, PINN, ENV_POLY02, 2, False),
    (F64, 3, 6, 5, SIN, DRM, ENV_POLY02, 149, False),
    (F64, 2, 2, 255, SIN, RAYLEIGH, (O.ENV_EXPWIN, 0.0, 2.0, ()), 7, False),
    (F64, 4, 8, 3, TANH, MSE, (O.ENV_NONE, 0.0, 2.0, ()), 1000, False),
    (F64, 2, 6, 256, SIN, DRM, (O.ENV_NONE, 0.0, 2.0, ()), 1, False),
    (F32, 1, 2, 256, SIN, PINN, ENV_POLY02, 149, True),
    (F32, 5, 2, 5, TANH, PINN, ENV_POLY02, 1000, False),
    (F32, 5, 6, 3, SIN, PINN, ENV_POLY02, 7, True),
    (F32, 2, 6, 1, SIN, DRM, ENV_POLY02, 2, False),
    (F32, 3, 8, 5, TANH, MSE, ENV_POLY02, 1, False),
    (F32, 1, 3, 256, TANH, RAYLEIGH, ENV_POLY02, 1000, False),
    (F32, 2, 8, 255, SIN, DRM, (O.ENV_EXPWIN, 0.0, 2.0, ()), 149, False),
    # FLUX: one point per face (N = 2d), a single face (149 is prime), five and eight faces of 1000 points
    (F64, 5, 8, 256, TANH, FLUX, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(8), (), _cheb(3))), 10, False),
    (F32, 2, 2, 1, SIN, FLUX, ENV_NONE02, 149, False),
    (F64, 3, 2, 3, TANH, FLUX, (O.ENV_POLY, -2.0, 2.0, (_cheb(8), [0.5])), 1000, False),
    (F32, 4, 8, 255, SIN, FLUX, ENV_NONE02, 1000, False),
    # RITZ: f = NULL (g = alpha) at odd N
    (F64, 5, 8, 256, SIN, RITZ, (O.ENV_POLY, 0.0, 2.0, ((), _cheb(8, 0.0, 2.0))), 1000, False),
    (F32, 3, 2, 1, TANH, RITZ, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(3), _cheb(8), ())), 1000, False),
    (F64, 1, 8, 3, TANH, RITZ, ENV_POLY02, 1, False),
    (F32, 2, 2, 255, SIN, RITZ, ENV_NONE02, 7, False),
    # PARABOLIC: no envelope (the library refuses one)
    (F64, 5, 8, 256, SIN, PARABOLIC, ENV_NONE02, 7, True),
    (F64, 2, 2, 1, TANH, PARABOLIC, ENV_NONE02, 1000, True),
    (F32, 3, 8, 3, SIN, PARABOLIC, ENV_NONE02, 1, False),
    (F32, 4, 2, 255, TANH, PARABOLIC, ENV_NONE02, 1000, True),
]


def _ids(cases):
    return ["-".join(str(v).replace("torch.", "") for v in (c[0], f"d{c[1]}", f"nl{c[2]}", f"H{c[3]}", NAME[c[5]],
                                                             f"n{c[7]}")) for c in cases]


def _flux_mask(d, N):
    """The face mask with the most faces whose count divides N (of those, the top bits): a FLUX batch of N points is
    popcount(mask) equal blocks."""
    p = max(k for k in range(1, 2 * d + 1) if N % k == 0)
    return ((1 << 2 * d) - 1) ^ ((1 << (2 * d - p)) - 1)


def _on_faces(X, faces, lo, hi):
    """Puts each block of a FLUX batch on its face: the face coordinate of the block's points set to lo or hi."""
    ax, s = O.face_blocks(faces, X.shape[0])
    X[np.arange(X.shape[0]), ax] = np.where(s > 0, hi, lo)
    return X


def _case(dtype, d, nl, H, act, kind, env, N, energy_ptr, seed=0):
    """One call of program `kind`.  PINN, DRM and MSE get white-noise f, PINN and RAYLEIGH per-point beta.  FLUX, RITZ
    and PARABOLIC get one-signed f (see test_tc_tile_edges_vs_oracle for why): FLUX on the faces of _flux_mask(d, N)
    with a per-point Robin beta on tanh nets and a constant one on sin nets; RITZ with beta >= 0 chosen the same way and
    f = NULL (g = alpha) when N is odd; PARABOLIC with alpha < 0, per-point beta and no envelope."""
    rng = np.random.default_rng(seed + 1000 * d + 10 * nl + H + N)
    Ws, bs = _rand_net(rng, d, H, nl, dtype)
    net = _Net(Ws, bs, act, dtype)
    kind_e, lo, hi, nodes = env
    X = _points(rng, N, d, lo + 0.05 * (hi - lo), hi - 0.05 * (hi - lo))
    f = rng.normal(size=N) if kind in (PINN, DRM, MSE) else None
    beta = rng.uniform(0.5, 1.5, N) if kind in (PINN, RAYLEIGH) else None
    alpha = {PINN: -0.5, DRM: 0.5, RAYLEIGH: 0.75, MSE: 1.0, FLUX: 0.75, RITZ: -1.25, PARABOLIC: -0.375}[kind]
    beta_const, faces = 0.0, 0
    if kind in (FLUX, RITZ, PARABOLIC):
        f = rng.uniform(1.0, 2.0, N)
        if kind == PARABOLIC:
            assert kind_e == O.ENV_NONE and not nodes, "PARABOLIC takes no envelope"
            beta = rng.uniform(0.5, 1.5, N)
        elif act == TANH:
            beta = rng.uniform(0.0 if kind == RITZ else 0.5, 1.5, N)
        else:
            beta_const = 0.8
        if kind == RITZ and N % 2:
            f = None
        if kind == FLUX:
            faces = _flux_mask(d, N)
            X = _on_faces(X, faces, lo, hi)
    return _Case(net, _envelope(kind_e, lo, hi, nodes, dtype), kind, X, alpha=alpha, f=f, beta=beta,
                 beta_const=beta_const, E=0.375, energy_ptr=energy_ptr, faces=faces)


@pytest.mark.parametrize("dtype,d,nl,H,act,kind,env,N,energy_ptr", GENERIC, ids=_ids(GENERIC))
def test_generic_kernel_at_the_edges_vs_oracle(dtype, d, nl, H, act, kind, env, N, energy_ptr):
    case = _case(dtype, d, nl, H, act, kind, env, N, energy_ptr)
    with _path("simt"):
        got = case.run()
    assert got["path"] == 0
    _assert_matches_oracle(case, got, case.oracle(), f"generic {case.net.c.dim}-D nl{nl} H{H} n{N}")


@pytest.mark.parametrize("order", [0, 1, 2])
@pytest.mark.parametrize("dtype", [F64, F32], ids=["float64", "float32"])
def test_generic_kernel_launches_its_largest_tiles(dtype, order):
    """With 64 points per SM the generic kernel's plan takes the largest point tile that shared memory and the block
    size of the kernel allow, which the point counts above rarely reach.  Every dim at widths of 25, 50 and 64 thread
    groups per point (H = 100, 200, 256) must launch there and match the oracle.  (The fp32 order-2 4-D kernel uses 197
    registers: a plan that sized its blocks from the register count alone picked 320 threads, which do not launch.)"""
    kind = {0: MSE, 1: DRM, 2: PINN}[order]
    N = 64 * _sms()
    for d in range(1, 6):
        for H in (100, 200, 256):
            case = _case(dtype, d, 2, H, TANH, kind, ENV_POLY02, N, False, seed=7)
            with _path("simt"):
                got = case.run()
            assert got["path"] == 0
            _assert_matches_oracle(case, got, case.oracle(), f"generic {NAME[kind]} {d}-D H{H} n{N}")


# dtype, d, n_linear, H, activation, order, N
JETS = [(F64, 5, 8, 256, SIN, 2, 7), (F64, 1, 2, 1, TANH, 2, 149), (F64, 3, 6, 255, SIN, 1, 2), (F64, 2, 7, 3, TANH, 0, 1000),
        (F32, 1, 2, 256, SIN, 2, 149), (F32, 5, 8, 5, TANH, 1, 7), (F32, 4, 6, 1, SIN, 0, 1), (F32, 2, 3, 255, SIN, 2, 1000)]


@pytest.mark.parametrize("dtype,d,nl,H,act,order,N", JETS)
def test_generic_jets_at_the_edges_vs_oracle(dtype, d, nl, H, act, order, N):
    """pde_jets_forward / pde_jets_backward on the generic kernel: jets and the reverse sweep of arbitrary cotangents."""
    L, lib = _lib()
    rng = np.random.default_rng(7 * d + nl + H + N)
    Ws, bs = _rand_net(rng, d, H, nl, dtype)
    net = _Net(Ws, bs, act, dtype)
    X = _rnd(rng.uniform(0, 2, (N, d)), dtype)
    Ch = 1 + order * d
    Jbar = _rnd(rng.normal(size=(N, Ch)), dtype)
    J, cache = O.mlp_jets_forward(Ws, bs, X, act, order)
    gWs, gbs = O.mlp_jets_backward(Ws, bs, cache, Jbar)
    with _path("simt"):
        got_J, got_g, _ = _run_jets(net, order, X, Jbar, POISON)
        assert lib.pde_last_kernel_path() == 0
    tol = _tol(dtype)
    Jg = got_J.double().cpu().numpy().reshape(N, Ch)
    assert np.max(np.abs(Jg - J)) <= 5 * tol * max(1.0, np.abs(J).max())
    assert_grads_close(net.unflat(got_g), (gWs, gbs), tol, f"jets d{d} nl{nl} H{H} order{order}")


def _run_jets(net, order, X, Jbar, fill):
    """pde_jets_forward then pde_jets_backward on buffers filled with `fill`; checks that nothing is written past the ends."""
    L, lib = _lib()
    dt = net.dtype
    N, d = X.shape
    Ch = 1 + order * d
    Xd, Jbd = _dev(X, dt), _dev(Jbar, dt)
    ws = _workspace(net, order, N, fill)
    J = _buf(N * Ch, dt, fill)
    L.check(lib.pde_jets_forward(C.byref(net.c), order, Xd.data_ptr(), N, J.data_ptr(), ws.data_ptr(), ws.numel(), _stream()),
            "pde_jets_forward")
    path_fwd = lib.pde_last_kernel_path()
    ws.fill_(fill)
    g = _buf(net.n_params, dt, fill)
    L.check(lib.pde_jets_backward(C.byref(net.c), order, Xd.data_ptr(), N, Jbd.data_ptr(), g.data_ptr(), ws.data_ptr(),
                                  ws.numel(), _stream()), "pde_jets_backward")
    assert lib.pde_last_kernel_path() == path_fwd
    torch.cuda.synchronize()
    assert _untouched_tail(J, N * Ch, fill) and _untouched_tail(g, net.n_params, fill)
    return J[:N * Ch], g[:net.n_params], path_fwd


# ================================================================================================ (c) tensor-core kernel
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# d, n_linear, H, activation, program, envelope, N, energy through the pointer, seed
TC = [
    # trainable energy: dE through the fused kernel's reduction (d = 2, 3) and the 5-D split's pointwise kernel
    (2, 5, 64, SIN, PINN, ENV_POLY02, 1000, True, None),
    (3, 4, 40, TANH, PINN, (O.ENV_EXPWIN, -2.0, 2.0, ()), 777, True, None),
    (5, 5, 64, SIN, PINN, ENV_POLY02, 1500, True, None),
    # forced nodes on the fused kernel: PDE_MAX_NODES on one dimension, nodes on several
    (1, 5, 64, SIN, PINN, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(8),)), 2000, False, None),
    (3, 5, 64, TANH, RAYLEIGH, (O.ENV_NONE, -2.0, 2.0, (_cheb(3), (), _cheb(8))), 1500, False, None),
    (4, 3, 64, SIN, PINN, (O.ENV_POLY, -2.0, 2.0, (_cheb(2), _cheb(8), [0.25], _cheb(5))), 1200, True, None),
    (3, 5, 64, SIN, DRM, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(8), _cheb(8), _cheb(8))), 900, False, None),
    # the 5-D split with everything it evaluates on its own: EXPWIN, nodes, per-point beta, energy pointer, seed
    (5, 4, 48, TANH, PINN, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(2), (), _cheb(8), [0.5], _cheb(3))), 3000, True, [0.3]),
    (5, 5, 64, SIN, PINN, (O.ENV_POLY, -2.0, 2.0, ((), _cheb(4))), 700, False, [-1.75]),
    # the fused residual step at width 1 and one unit below a full K-chunk
    (3, 4, 1, SIN, PINN, ENV_POLY02, 1000, True, None),
    (2, 3, 63, TANH, PINN, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(3), ())), 1500, True, [0.3]),
    (3, 5, 1, TANH, DRM, ENV_POLY02, 1000, False, None),
    (4, 4, 63, SIN, DRM, ENV_POLY02, 800, False, [-1.75]),
    # FLUX (order 1): narrow and odd widths, 2..4 hidden layers, nodes, the face walk across tiles and CTAs
    (3, 3, 1, SIN, FLUX, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(8), (), _cheb(3))), 1200, False, None),
    (2, 4, 17, TANH, FLUX, (O.ENV_POLY, -2.0, 2.0, (_cheb(5), [0.25])), 1000, False, [0.3]),
    (4, 5, 63, SIN, FLUX, ENV_NONE02, 777, False, None),
    (1, 5, 64, TANH, FLUX, ENV_POLY02, 2000, False, [-1.75]),
    (5, 3, 3, TANH, FLUX, ENV_NONE02, 4000, False, None),
    # RITZ (order 0)
    (3, 3, 3, TANH, RITZ, (O.ENV_POLY, -2.0, 2.0, (_cheb(8), _cheb(2), ())), 1500, False, None),
    (5, 4, 63, SIN, RITZ, (O.ENV_EXPWIN, -2.0, 2.0, ((), _cheb(4), (), (), _cheb(8))), 999, False, [0.3]),
    (2, 5, 1, TANH, RITZ, ENV_NONE02, 2000, False, None),
    (4, 3, 17, SIN, RITZ, ENV_POLY02, 777, False, [-1.75]),
    (1, 4, 64, TANH, RITZ, (O.ENV_EXPWIN, -2.0, 2.0, (_cheb(8),)), 1001, False, None),
    # PARABOLIC (the NLAP = d - 1 instantiations), energy through the pointer
    (2, 3, 1, TANH, PARABOLIC, ENV_NONE02, 1000, True, None),
    (3, 4, 63, SIN, PARABOLIC, ENV_NONE02, 1500, True, [0.3]),
    (4, 5, 17, TANH, PARABOLIC, ENV_NONE02, 2000, True, None),
    (3, 5, 3, SIN, PARABOLIC, ENV_NONE02, 777, True, [-1.75]),
    (2, 4, 64, SIN, PARABOLIC, ENV_NONE02, 3000, False, None),
    (4, 3, 64, TANH, PARABOLIC, ENV_NONE02, 1200, True, [0.3]),
]


@pytest.mark.parametrize("d,nl,H,act,kind,env,N,energy_ptr,seed", TC)
def test_tc_options_vs_oracle(d, nl, H, act, kind, env, N, energy_ptr, seed):
    case = _case(F32, d, nl, H, act, kind, env, N, energy_ptr, seed=1)
    with _path("tc"):
        assert case.query_path() == 1
        got = case.run(seed=seed)
    assert got["path"] == 1
    _assert_matches_oracle(case, got, case.oracle(seed=seed), f"tc {d}-D nl{nl} H{H} n{N}")


TILE_EDGES = {"1": lambda sms: 1, "63": lambda sms: 63, "64": lambda sms: 64, "65": lambda sms: 65,
              "sms*64-1": lambda sms: sms * 64 - 1, "sms*64+1": lambda sms: sms * 64 + 1}


@pytest.mark.parametrize("d", [3, 5])
@pytest.mark.parametrize("tiles", list(TILE_EDGES))
def test_tc_tile_edges_vs_oracle(d, tiles):
    """Point counts at the 64-point tile edges and one past a full wave of CTAs (one tile per SM), on the fused kernel
    (d = 3) and the 5-D split (whose pointwise kernel runs 256-point blocks).

    The tail itself is checked exactly: one more point with two coordinates on the boundary and f = 0 contributes
    nothing to any output, so appending it (which fills or opens a tile) must leave sums, gradient and dE bit-identical.
    The oracle comparison uses the reference workload's right-hand side (Poisson_ND.py:49-58, one-signed on the box).
    With white-noise f the output-bias gradient is a signed sum over the points: at 63 points a draw where it cancels
    374-fold puts the tensor-core kernel's 3-term fp16 operand splits at 4.5e-5 from the oracle, whatever the tail."""
    N = TILE_EDGES[tiles](_sms())
    rng = np.random.default_rng(2 + 1000 * d + N)
    Ws, bs = _rand_net(rng, d, 64, 5, F32)
    net = _Net(Ws, bs, SIN, F32)
    X = _rnd(_points(rng, N, d), F32)
    f = d * (math.pi / 2) ** 2 * np.prod(np.sin(math.pi * X / 2), axis=1)
    beta = rng.uniform(0.5, 1.5, N)
    env = _envelope(O.ENV_POLY, 0.0, 2.0, (), F32)
    case = _Case(net, env, PINN, X, alpha=-0.5, f=f, beta=beta, E=0.375, energy_ptr=True)
    inert = np.ones((1, d))
    inert[0, :2] = 0.0
    padded = _Case(net, env, PINN, np.concatenate([X, inert]), alpha=-0.5, f=np.append(f, 0.0), beta=np.append(beta, 1.0),
                   E=0.375, energy_ptr=True)
    with _path("tc"):
        got = case.run()
        more = padded.run(inv_n=1.0 / N)
    assert got["path"] == more["path"] == 1
    for k, n in (("sums", 1), ("grad", net.n_params), ("dE", 1)):
        assert torch.equal(_bytes(more[k], n), _bytes(got[k], n)), k
    _assert_matches_oracle(case, got, case.oracle(), f"tc {d}-D n{N}")


@pytest.mark.parametrize("tiles", list(TILE_EDGES))
@pytest.mark.parametrize("kind", [RITZ, FLUX, PARABOLIC], ids=[NAME[k] for k in (RITZ, FLUX, PARABOLIC)])
def test_tc_tile_edges_of_the_boundary_and_parabolic_programs_vs_oracle(kind, tiles):
    """The tile edges of test_tc_tile_edges_vs_oracle at d = 3 for RITZ, FLUX and PARABOLIC, with one-signed data.

    RITZ keeps the exact tail check: the appended point has two coordinates on the POLY boundary and f = 0, so u = 0 and
    its cotangent beta u - f is 0.  FLUX runs on the mask with the most faces whose count divides N (N follows the SM
    count and may be prime; the mask is in every message), and PARABOLIC without an envelope; for those two a point
    more would change the face layout or contribute, so they are compared with the oracle only."""
    d = 3
    N = TILE_EDGES[tiles](_sms())
    rng = np.random.default_rng(20 + kind + 1000 * d + N)
    Ws, bs = _rand_net(rng, d, 64, 5, F32)
    net = _Net(Ws, bs, TANH, F32)
    faces = _flux_mask(d, N) if kind == FLUX else 0
    env = _envelope(O.ENV_NONE if kind == PARABOLIC else O.ENV_POLY, 0.0, 2.0, (), F32)
    X = _points(rng, N, d)
    if kind == FLUX:
        X = _on_faces(X, faces, 0.0, 2.0)
    f, beta = rng.uniform(1.0, 2.0, N), rng.uniform(0.5, 1.5, N)
    alpha = {RITZ: -1.25, FLUX: 0.75, PARABOLIC: -0.375}[kind]
    case = _Case(net, env, kind, X, alpha=alpha, f=f, beta=beta, E=0.375, energy_ptr=True, faces=faces)
    what = f"tc {NAME[kind]} {d}-D n{N} faces={faces:#b}"
    with _path("tc"):
        got = case.run()
        if kind == RITZ:
            inert = np.ones((1, d))
            inert[0, :2] = 0.0
            padded = _Case(net, env, kind, np.concatenate([X, inert]), alpha=alpha, f=np.append(f, 0.0),
                           beta=np.append(beta, 1.0), E=0.375, energy_ptr=True)
            more = padded.run(inv_n=1.0 / N)
            assert more["path"] == 1
            for k, n in (("sums", 1), ("grad", net.n_params), ("dE", 1)):
                assert torch.equal(_bytes(more[k], n), _bytes(got[k], n)), k
    assert got["path"] == 1, what
    _assert_matches_oracle(case, got, case.oracle(), what)


# n_linear, H, expected family at 8192 points (automatic choice)
DECLINE = [(3, 64, 1), (5, 64, 1), (2, 64, 0), (6, 64, 0), (4, 65, 0)]


@pytest.mark.parametrize("nl,H,family", DECLINE)
def test_tc_decline_edges(nl, H, family):
    """The tensor-core kernel takes fp32 nets of 2..4 hidden layers up to width 64; one layer fewer or more, or one unit
    wider, and the generic kernel serves the call — pde_query_path says so beforehand, the launch reports it, and both
    match the oracle."""
    case = _case(F32, 2, nl, H, TANH, PINN, ENV_POLY02, 8192, False, seed=3)
    with _path("auto"):
        assert case.query_path() == family
        got = case.run()
    assert got["path"] == family
    _assert_matches_oracle(case, got, case.oracle(), f"auto nl{nl} H{H}")


# d, n_linear, H, expected family at 8192 points (automatic choice)
PARABOLIC_DECLINE = [(3, 4, 64, 1), (2, 2, 64, 0), (2, 6, 64, 0), (2, 4, 65, 0), (5, 4, 64, 0)]


@pytest.mark.parametrize("d,nl,H,family", PARABOLIC_DECLINE)
def test_tc_decline_edges_of_the_parabolic_program(d, nl, H, family):
    """PARABOLIC declines like PINN (one hidden layer, five, or width 65) and also at d = 5, where the tensor-core
    kernel has no split pass for it: the generic kernel serves those calls and every call matches the oracle."""
    case = _case(F32, d, nl, H, SIN, PARABOLIC, ENV_NONE02, 8192, True, seed=3)
    with _path("auto"):
        assert case.query_path() == family
        got = case.run()
    assert got["path"] == family
    _assert_matches_oracle(case, got, case.oracle(), f"auto parabolic d{d} nl{nl} H{H}")


# ================================================================================================ (d) seed and inv_n
# family, dtype, d, n_linear, H, program, N, seed
LINEAR = [("simt", F64, 2, 3, 20, RAYLEIGH, 500, [0.3, -2.0]), ("simt", F32, 1, 4, 33, PINN, 300, [0.3]),
          ("tc", F32, 3, 5, 64, PINN, 5000, [0.3]), ("tc", F32, 2, 4, 64, RAYLEIGH, 3000, [0.3, -2.0]),
          ("tc", F32, 5, 5, 64, PINN, 2000, [0.3]),
          ("simt", F64, 3, 4, 20, FLUX, 600, [0.3]), ("simt", F32, 2, 3, 33, RITZ, 300, [-2.0]),
          ("simt", F64, 3, 3, 20, PARABOLIC, 500, [0.3]), ("tc", F32, 3, 5, 64, FLUX, 3000, [0.3]),
          ("tc", F32, 2, 4, 17, RITZ, 3000, [-2.0]), ("tc", F32, 3, 4, 64, PARABOLIC, 5000, [0.3])]


@pytest.mark.parametrize("family,dtype,d,nl,H,kind,N,seed", LINEAR)
def test_seed_and_inv_n_are_linear(family, dtype, d, nl, H, kind, N, seed):
    """With a seed s and an arbitrary inv_n the gradient and dE are inv_n n sum_k s_k (those of seed e_k, inv_n = 1/n),
    the NULL seed is the all-ones seed, and the sums do not depend on either, bit for bit."""
    case = _case(dtype, d, nl, H, SIN, kind, ENV_NONE02 if kind == PARABOLIC else ENV_POLY02, N,
                 kind in (PINN, PARABOLIC), seed=4)
    inv_n = 0.625 / N
    K = NQ[kind]
    with _path(family):
        base = case.run()
        units = [case.run(seed=list(np.eye(K)[k])) for k in range(K)]
        got = case.run(seed=seed, inv_n=inv_n)
    assert base["path"] == got["path"] == (1 if family == "tc" else 0)
    tol = _tol(dtype)
    s = _rnd(seed, dtype)
    for r in units + [got]:
        assert torch.equal(_bytes(r["sums"], K), _bytes(base["sums"], K))
    g = [u["grad"].double() for u in units]
    scale = max(float(x.abs().max()) for x in g)
    assert float((sum(g) - base["grad"].double()).abs().max()) <= tol * scale
    want = inv_n * N * sum(float(sk) * gk for sk, gk in zip(s, g))
    assert float((got["grad"].double() - want).abs().max()) <= tol * scale * inv_n * N * max(abs(s))
    if kind in (PINN, PARABOLIC):
        dE1 = float(units[0]["dE"][0])
        assert float(base["dE"][0]) == pytest.approx(dE1, rel=tol, abs=0)
        assert float(got["dE"][0]) == pytest.approx(inv_n * N * float(s[0]) * dE1, rel=tol, abs=0)


# ================================================================================================ (e) output contract
# family, dtype, d, n_linear, H, program, N
CONTRACT = [("simt", F64, 2, 3, 20, PINN, 300), ("simt", F32, 1, 4, 256, RAYLEIGH, 149), ("tc", F32, 3, 5, 64, PINN, 1000),
            ("tc", F32, 2, 4, 64, RAYLEIGH, 5000), ("tc", F32, 5, 5, 64, PINN, 500),
            ("simt", F64, 3, 4, 20, FLUX, 300), ("simt", F32, 2, 8, 256, RITZ, 149), ("simt", F64, 4, 3, 20, PARABOLIC, 300),
            ("tc", F32, 3, 5, 64, FLUX, 996), ("tc", F32, 2, 3, 63, RITZ, 1000), ("tc", F32, 3, 4, 64, PARABOLIC, 1000)]


@pytest.mark.parametrize("family,dtype,d,nl,H,kind,N", CONTRACT)
def test_residual_outputs_and_workspace_carry_no_state(family, dtype, d, nl, H, kind, N):
    """sums, grad and energy_grad are pure outputs and the workspace holds nothing across calls: with every byte of
    them NaN beforehand the results are bit-identical to a run on zeroed buffers, nothing past their ends is written,
    grad = NULL with energy_grad set still gives the same dE and sums (that call still runs the reverse sweep), and the
    sums-only call (grad and energy_grad NULL, no reverse sweep) gives the same sums."""
    case = _case(dtype, d, nl, H, TANH, kind, ENV_NONE02 if kind == PARABOLIC else ENV_POLY02, N,
                 kind in (PINN, PARABOLIC), seed=5)
    K = NQ[kind]
    with _path(family):
        clean = case.run(fill=0)
        dirty = case.run(fill=POISON)
        no_grad = case.run(fill=POISON, grad=False)
        sums_only = case.run(fill=POISON, grad=False, dE=False)
    assert clean["path"] == dirty["path"] == no_grad["path"] == sums_only["path"] == (1 if family == "tc" else 0)
    assert clean["intact"] and dirty["intact"] and no_grad["intact"] and sums_only["intact"]
    for k, n in (("sums", K), ("grad", case.net.n_params), ("dE", 1)):
        assert torch.equal(_bytes(dirty[k], n), _bytes(clean[k], n)), k
    assert torch.equal(_bytes(no_grad["sums"], K), _bytes(clean["sums"], K))
    assert torch.equal(_bytes(no_grad["dE"], 1), _bytes(clean["dE"], 1))
    assert torch.equal(_bytes(sums_only["sums"], K), _bytes(clean["sums"], K))
    assert torch.isfinite(clean["grad"]).all() and torch.isfinite(clean["sums"]).all()


@pytest.mark.parametrize("kind", [RITZ, FLUX, PARABOLIC, PINN, DRM], ids=[NAME[k] for k in (RITZ, FLUX, PARABOLIC, PINN, DRM)])
def test_tc_sums_only_call_over_three_tiles_per_cta(kind):
    """Without grad and energy_grad the tensor-core kernel runs forward only, and the two-slot W plan has to bring the
    first hidden layer's weights back for every tile by itself: over three tiles per CTA (and a tail) the sums must be
    bit-identical to the training call's — for the order-0 RITZ and order-1 FLUX branches, the PARABOLIC (NLAP = d - 1)
    instantiation and, at these widths, PINN and DRM."""
    N = 64 * _sms() * 3 + 29
    env = ENV_NONE02 if kind == PARABOLIC else ENV_POLY02
    case = _case(F32, 3, 5, 64, SIN, kind, env, N, kind in (PINN, PARABOLIC), seed=9)
    with _path("tc"):
        train = case.run(fill=POISON)
        sums_only = case.run(fill=POISON, grad=False, dE=False)
    assert train["path"] == sums_only["path"] == 1
    assert train["intact"] and sums_only["intact"]
    assert torch.isfinite(train["sums"]).all() and torch.isfinite(train["grad"]).all()
    assert torch.equal(_bytes(sums_only["sums"], 1), _bytes(train["sums"], 1)), (float(sums_only["sums"][0]),
                                                                                  float(train["sums"][0]))


@pytest.mark.parametrize("family,dtype,d,nl,H,order,N", [("simt", F64, 3, 4, 20, 2, 300), ("simt", F32, 2, 2, 256, 1, 149),
                                                          ("tc", F32, 2, 4, 64, 1, 700), ("tc", F32, 3, 5, 64, 0, 5000)])
def test_jets_outputs_and_workspace_carry_no_state(family, dtype, d, nl, H, order, N):
    """pde_jets_forward / pde_jets_backward: J and grad bit-identical whether their buffers and the workspace start as
    NaN bytes or zeros, nothing written past their ends."""
    rng = np.random.default_rng(6 + d + N)
    Ws, bs = _rand_net(rng, d, H, nl, dtype)
    net = _Net(Ws, bs, SIN, dtype)
    X = _rnd(rng.uniform(0, 2, (N, d)), dtype)
    Jbar = _rnd(rng.normal(size=(N, 1 + order * d)), dtype)
    with _path(family):
        Jc, gc, pc = _run_jets(net, order, X, Jbar, 0)
        Jd, gd, pd = _run_jets(net, order, X, Jbar, POISON)
    assert pc == pd == (1 if family == "tc" else 0)
    assert torch.equal(_bytes(Jd, Jd.numel()), _bytes(Jc, Jc.numel()))
    assert torch.equal(_bytes(gd, gd.numel()), _bytes(gc, gc.numel()))
    assert torch.isfinite(Jc).all() and torch.isfinite(gc).all()


# ================================================================================================ (g) ignored fields
def _same_outputs(a, b, n_params, what):
    for k, n in (("sums", 1), ("grad", n_params), ("dE", 1)):
        assert torch.equal(_bytes(a[k], n), _bytes(b[k], n)), f"{what}: {k}"


# family, dtype, d, n_linear, H, N
IGNORED = [("simt", F64, 3, 3, 20, 300), ("tc", F32, 3, 4, 64, 1200)]


@pytest.mark.parametrize("family,dtype,d,nl,H,N", IGNORED, ids=[c[0] for c in IGNORED])
@pytest.mark.parametrize("kind", [FLUX, RITZ], ids=[NAME[k] for k in (FLUX, RITZ)])
def test_energy_fields_are_ignored_by_flux_and_ritz(kind, family, dtype, d, nl, H, N):
    """FLUX and RITZ ignore the energy fields and have dq/dE = 0: with `energy` pointing at NaN and energy_const = NaN,
    sums and grad are bit-identical to a call with energy = NULL, and energy_grad is written as exactly 0 over a
    NaN-filled buffer."""
    case = _case(dtype, d, nl, H, TANH, kind, ENV_POLY02, N, False, seed=11)
    with _path(family):
        base = case.run(fill=POISON)
        nan = _dev(np.array([np.nan]), dtype)
        case.prog.energy, case.prog.energy_const = nan.data_ptr(), float("nan")
        got = case.run(fill=POISON)
    assert base["path"] == got["path"] == (1 if family == "tc" else 0)
    assert got["intact"]
    for k, n in (("sums", 1), ("grad", case.net.n_params)):
        assert torch.equal(_bytes(got[k], n), _bytes(base[k], n)), k
    assert float(got["dE"][0]) == 0.0 and float(base["dE"][0]) == 0.0, (float(got["dE"][0]), float(base["dE"][0]))


@pytest.mark.parametrize("family,dtype,d,nl,H,N", IGNORED, ids=[c[0] for c in IGNORED])
@pytest.mark.parametrize("kind", [PINN, RITZ, PARABOLIC], ids=[NAME[k] for k in (PINN, RITZ, PARABOLIC)])
def test_face_mask_is_ignored_by_every_program_but_flux(kind, family, dtype, d, nl, H, N):
    """`faces` is read by FLUX alone: a mask of 0x155 (not even a valid mask at d = 3) leaves sums, grad and dE
    bit-identical to faces = 0."""
    env = ENV_NONE02 if kind == PARABOLIC else ENV_POLY02
    case = _case(dtype, d, nl, H, SIN, kind, env, N, kind != RITZ, seed=12)
    with _path(family):
        base = case.run(fill=POISON)
        case.prog.faces = 0x155
        got = case.run(fill=POISON)
    assert base["path"] == got["path"] == (1 if family == "tc" else 0)
    assert got["intact"]
    _same_outputs(got, base, case.net.n_params, f"{NAME[kind]} faces=0x155")


@pytest.mark.parametrize("family,dtype,d,nl,H,N", IGNORED, ids=[c[0] for c in IGNORED])
def test_ritz_constant_g_is_alpha(family, dtype, d, nl, H, N):
    """RITZ with f = NULL uses g = alpha: bit-identical to f = an array of that constant (with alpha = NaN, which a
    call with f must not read)."""
    c = -1.25
    base = _case(dtype, d, nl, H, TANH, RITZ, ENV_POLY02, N + 1, False, seed=13)     # N + 1 odd: f = NULL
    assert base.f is None
    base.prog.alpha = c
    with_f = _Case(base.net, (base.env_c, base.env), RITZ, base.X, alpha=float("nan"), f=np.full(base.n, c), beta=base.beta,
                   beta_const=base.beta_const, E=base.E)
    with _path(family):
        a = base.run(fill=POISON)
        b = with_f.run(fill=POISON)
    assert a["path"] == b["path"] == (1 if family == "tc" else 0)
    assert a["intact"] and b["intact"]
    _same_outputs(a, b, base.net.n_params, "f = NULL, alpha = c vs f = c")
    assert torch.isfinite(a["grad"]).all() and torch.isfinite(a["sums"]).all()


# ================================================================================================ (f) WAN pointwise
class _Wan:
    """One pde_wan_pointwise problem on given network jets Ju, Jv (n, 1+d): both envelopes, the bump on [w_lo, w_hi]."""

    def __init__(self, dtype, X, Ju, Jv, w_lo, w_hi, eps_den, f, beta, E, alpha, env_u, env_v):
        L, _ = _lib()
        self.dtype, self.n, self.d = dtype, X.shape[0], X.shape[1]
        self.X, self.Ju, self.Jv = _rnd(X, dtype), _rnd(Ju, dtype), _rnd(Jv, dtype)
        self.f, self.beta = _rnd(f, dtype).reshape(-1, 1), _rnd(beta, dtype).reshape(-1, 1)
        self.E, self.alpha, self.w_lo, self.w_hi, self.eps_den = E, alpha, w_lo, w_hi, eps_den
        self.env_u, self.env_v = env_u, env_v
        self.Xd, self.Jud, self.Jvd = _dev(self.X, dtype), _dev(self.Ju, dtype), _dev(self.Jv, dtype)
        self.fd, self.bd, self.Ed = _dev(self.f.reshape(-1), dtype), _dev(self.beta.reshape(-1), dtype), _dev([E], dtype)
        w = L.Wan()
        w.dtype, w.dim = (L.F64 if dtype == F64 else L.F32), self.d
        w.alpha, w.beta_const, w.energy_const, w.w_lo, w.w_hi, w.eps_den = alpha, 0.0, 0.0, w_lo, w_hi, eps_den
        w.f, w.beta, w.energy = self.fd.data_ptr(), self.bd.data_ptr(), self.Ed.data_ptr()
        w.env_u, w.env_v = env_u[0], env_v[0]
        self.c = w

    def run(self, seed, inv_n, fill):
        L, lib = _lib()
        Ch = 1 + self.d
        sums = _buf(5, self.dtype, fill)
        Jbu, Jbv = _buf(self.n * Ch, self.dtype, fill), _buf(self.n * Ch, self.dtype, fill)
        ws = torch.full((max(1 << 16, 8 * 8 * 4 * _sms()),), fill, dtype=torch.uint8, device="cuda")
        sd = _dev(_rnd(seed, self.dtype), self.dtype)
        rc = lib.pde_wan_pointwise(C.byref(self.c), self.Xd.data_ptr(), self.n, self.Jud.data_ptr(), self.Jvd.data_ptr(),
                                   sd.data_ptr(), inv_n, sums.data_ptr(), Jbu.data_ptr(), Jbv.data_ptr(), ws.data_ptr(),
                                   ws.numel(), _stream())
        L.check(rc, "pde_wan_pointwise")
        torch.cuda.synchronize()
        assert _untouched_tail(sums, 5, fill) and _untouched_tail(Jbu, self.n * Ch, fill) and _untouched_tail(Jbv, self.n * Ch, fill)
        return sums[:5], Jbu[:self.n * Ch].view(self.n, Ch), Jbv[:self.n * Ch].view(self.n, Ch)

    def oracle(self, seed, inv_n):
        """The per-point quantities of oracle/jets_numpy.wan_means on these jets: sums of q0..q3 and dq0/dE, the
        cotangents sum_k seed_k inv_n dq_k/dJ of both networks' jets, and the terms' magnitudes for the bars."""
        d, X = self.d, self.X
        eu, ev = self.env_u[1], self.env_v[1]
        Uu, xu = O.apply_envelope(self.Ju, X, 1, eu["kind"], eu["lo"], eu["hi"], eu["nodes"])
        Uv, xv = O.apply_envelope(self.Jv, X, 1, ev["kind"], ev["lo"], ev["hi"], ev["nodes"])
        w, dw = O.bump_weight(X, self.w_lo, self.w_hi, self.eps_den)
        u, gu, v, gv = Uu[:, 0:1], Uu[:, 1:], Uv[:, 0:1], Uv[:, 1:]
        phi, gphi = w * v, dw * v + w * gv
        bt, E, a, f = self.beta, self.E, self.alpha, self.f
        q = [a * np.sum(gu * gphi, axis=1, keepdims=True) + (bt - E) * u * phi - f * phi, phi * phi, u * u,
             np.sum(gv * gv, axis=1, keepdims=True) + v * v, -u * phi]
        s = _rnd(seed, self.dtype) * inv_n
        Ub, Vb = np.zeros_like(Uu), np.zeros_like(Uv)
        Ub[:, 0:1] = s[0] * (bt - E) * phi + s[2] * 2.0 * u
        Ub[:, 1:] = s[0] * a * gphi
        Vb[:, 0:1] = s[0] * (((bt - E) * u - f) * w + np.sum(a * gu * dw, axis=1, keepdims=True)) + s[1] * 2.0 * phi * w \
            + s[3] * 2.0 * v
        Vb[:, 1:] = s[0] * a * gu * w + s[3] * 2.0 * gv
        return ([float(np.sum(t)) for t in q], [float(np.sum(np.abs(t))) for t in q],
                O.envelope_backward(Ub, xu, 1, d), O.envelope_backward(Vb, xv, 1, d))


def _ulp_step(x, direction, dtype):
    return float(np.nextafter(np.float32(x), np.float32(direction))) if dtype == F32 else float(np.nextafter(x, direction))


def _bump_edge_points(rng, dtype, eps_den, w_lo, w_hi, centre, d):
    """Rows whose i-th coordinate sits at w_lo / w_hi, one ulp outside, one ulp and 1e-6 inside, at the centre or near
    the edge, the others drawn inside the box.  One ulp inside is left out in float64 with eps_den > 0: there
    1 - t^2 < eps_den and the bump's denominator changes sign (the reference's own weight is infinite)."""
    edge = []
    for b, out in ((w_lo, w_lo - 1.0), (w_hi, w_hi + 1.0)):
        edge += [b, _ulp_step(b, out, dtype), b + (centre - b) * 1e-6]
        if dtype == F32 or eps_den == 0.0:
            edge.append(_ulp_step(b, centre, dtype))
    h = 0.5 * (w_hi - w_lo)
    edge += [centre, centre + 0.999 * h, centre - 0.9 * h]
    rows = []
    for e in edge:
        for i in range(d):
            for _ in range(3):
                x = rng.uniform(w_lo + 0.2 * h, w_hi - 0.2 * h, d)
                x[i] = e
                rows.append(x)
    return np.array(rows)


@pytest.mark.parametrize("dtype", [F64, F32])
@pytest.mark.parametrize("eps_den", [0.0, 1e-10])
def test_wan_bump_edges_vs_oracle(dtype, eps_den):
    """pde_wan_pointwise at the edges of the bump's support (_bump_edge_points) and across it: sums and both networks'
    cotangents vs the per-point restatement of oracle/jets_numpy.wan_means (bump weight from bump_weight), itself
    checked against wan_means; NaN-filled outputs and workspace give the same bits as zeroed ones."""
    rng = np.random.default_rng(8)
    d, w_lo, w_hi = 2, -0.5, 1.5          # centre 0.5 and half-width 1: t = x - 0.5 exactly in both dtypes
    X = _rnd(np.concatenate([_bump_edge_points(rng, dtype, eps_den, w_lo, w_hi, 0.5, d), rng.uniform(-0.7, 1.7, (300, d))]),
             dtype)
    N = X.shape[0]
    (uW, ub), (vW, vb) = _rand_net(rng, d, 8, 3, dtype), _rand_net(rng, d, 8, 3, dtype)
    Ju, Jv = O.mlp_jets_forward(uW, ub, X, SIN, 1)[0], O.mlp_jets_forward(vW, vb, X, TANH, 1)[0]
    env_u = _envelope(O.ENV_POLY, -0.5, 1.5, (), dtype)
    env_v = _envelope(O.ENV_EXPWIN, -0.5, 1.5, ([0.25],), dtype)
    f, beta, E, alpha = rng.normal(size=N), rng.uniform(0.5, 1.5, N), 0.625, 0.75
    prob = _Wan(dtype, X, Ju, Jv, w_lo, w_hi, eps_den, f, beta, E, alpha, env_u, env_v)
    seed, inv_n = [0.5, -1.25, 2.0, 0.75], 1.0 / N
    sums, Jbu, Jbv = prob.run(seed, inv_n, POISON)
    s_c, Jbu_c, Jbv_c = prob.run(seed, inv_n, 0)
    assert torch.equal(_bytes(sums, 5), _bytes(s_c, 5))
    assert torch.equal(_bytes(Jbu, Jbu.numel()), _bytes(Jbu_c, Jbu.numel()))
    assert torch.equal(_bytes(Jbv, Jbv.numel()), _bytes(Jbv_c, Jbv.numel()))
    want, scales, Ubar, Vbar = prob.oracle(seed, inv_n)
    if dtype == F64:     # the restatement is wan_means, point by point
        means, Gu, Gv, dE = O.wan_means({"Ws": uW, "bs": ub, "act": SIN, "env": env_u[1]},
                                        {"Ws": vW, "bs": vb, "act": TANH, "env": env_v[1]}, X, prob.f, w_lo, w_hi,
                                        a=alpha, beta=prob.beta, E=E, eps_den=eps_den)
        assert np.allclose(np.array(want) / N, means + [dE], rtol=1e-12, atol=0)
    tol = _tol(dtype)
    got = sums.double().cpu().numpy()
    for k in range(5):
        assert abs(got[k] - want[k]) <= tol * max(scales[k], 1e-300), (k, got[k], want[k])
    for name, g, ww in (("Jbar_u", Jbu, Ubar), ("Jbar_v", Jbv, Vbar)):
        g = g.double().cpu().numpy()
        assert np.isfinite(g).all(), name
        err = np.max(np.abs(g - ww), axis=0) / np.maximum(np.max(np.abs(ww), axis=0), 1e-300)
        assert err.max() <= tol, (name, err)
