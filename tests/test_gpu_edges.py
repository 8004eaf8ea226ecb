"""GPU parity tests of the C ABI at the edges of its advertised envelope (run with -m gpu on a B200).

include/pde_b200.h promises dim 1..5, 2..8 Linear layers, hidden widths 1..256, up to PDE_MAX_NODES forced nodes per
dimension, a trainable-energy pointer with its gradient, a free seed vector and inv_n, and any n >= 1.  The reference
shapes the other parity tests use stay well inside that envelope; here the ABI is driven directly through the ctypes
structs, every output buffer and the workspace belong to the test (so they can be poisoned), and the reference is the
float64 numpy oracle (oracle/jets_numpy).  The cases sit where kernels go wrong: one hidden layer, width 1 (padded to 8
units) and 256 (two warps per point, W streamed in K-chunks), the deepest net, tile tails, tensor-core options that the
reference shapes never reach, and the decline edges between the two kernel families.

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
PINN, DRM, RAYLEIGH, MSE = 1, 2, 3, 4
ORDER = {PINN: 2, DRM: 1, RAYLEIGH: 1, MSE: 0}
NQ = {PINN: 1, DRM: 1, RAYLEIGH: 2, MSE: 1}
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

    def __init__(self, net, env, kind, X, alpha=1.0, f=None, beta=None, beta_const=0.0, E=0.0, energy_ptr=False):
        L, _ = _lib()
        dt = net.dtype
        self.net, self.env_c, self.env = net, env[0], env[1]
        self.kind, self.alpha = kind, alpha
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
        p.kind, p.alpha, p.beta_const = kind, alpha, self.beta_const
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
    at one point and at 8192, with the kernel family chosen automatically and forced onto the tensor cores."""
    L, lib = _lib()
    progs = {0: MSE, 1: DRM, 2: PINN}
    refused = []
    for which in ("auto", "tc"):
        with _path(which):
            for dt in (L.F32, L.F64):
                for d in range(1, 6):
                    for order in range(3):
                        prog = L.Program()
                        prog.kind = progs[order]
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
                                    if rc != 0 or nb.value == 0 or path not in (0, 1):
                                        refused.append(("f64" if dt == L.F64 else "f32", f"d={d}", f"order={order}",
                                                        f"n_linear={nl}", f"H={H}", f"n={n}", which, rc, path))
    assert not refused, f"{len(refused)} shapes inside the header's envelope refused: {refused}"


# ================================================================================================ (b) generic kernel
# dtype, d, n_linear, H, activation, program, envelope (kind, lo, hi, nodes), N, energy through the pointer
ENV_POLY02 = (O.ENV_POLY, 0.0, 2.0, ())
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
]


def _ids(cases):
    return ["-".join(str(v).replace("torch.", "") for v in (c[0], f"d{c[1]}", f"nl{c[2]}", f"H{c[3]}",
                                                             {PINN: "pinn", DRM: "drm", RAYLEIGH: "ray", MSE: "mse"}[c[5]],
                                                             f"n{c[7]}")) for c in cases]


def _case(dtype, d, nl, H, act, kind, env, N, energy_ptr, seed=0):
    rng = np.random.default_rng(seed + 1000 * d + 10 * nl + H + N)
    Ws, bs = _rand_net(rng, d, H, nl, dtype)
    net = _Net(Ws, bs, act, dtype)
    kind_e, lo, hi, nodes = env
    X = _points(rng, N, d, lo + 0.05 * (hi - lo), hi - 0.05 * (hi - lo))
    f = rng.normal(size=N) if kind in (PINN, DRM, MSE) else None
    beta = rng.uniform(0.5, 1.5, N) if kind in (PINN, RAYLEIGH) else None
    alpha = {PINN: -0.5, DRM: 0.5, RAYLEIGH: 0.75, MSE: 1.0}[kind]
    return _Case(net, _envelope(kind_e, lo, hi, nodes, dtype), kind, X, alpha=alpha, f=f, beta=beta, E=0.375,
                 energy_ptr=energy_ptr)


@pytest.mark.parametrize("dtype,d,nl,H,act,kind,env,N,energy_ptr", GENERIC, ids=_ids(GENERIC))
def test_generic_kernel_at_the_edges_vs_oracle(dtype, d, nl, H, act, kind, env, N, energy_ptr):
    case = _case(dtype, d, nl, H, act, kind, env, N, energy_ptr)
    with _path("simt"):
        got = case.run()
    assert got["path"] == 0
    _assert_matches_oracle(case, got, case.oracle(), f"generic {case.net.c.dim}-D nl{nl} H{H} n{N}")


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


# ================================================================================================ (d) seed and inv_n
# family, dtype, d, n_linear, H, program, N, seed
LINEAR = [("simt", F64, 2, 3, 20, RAYLEIGH, 500, [0.3, -2.0]), ("simt", F32, 1, 4, 33, PINN, 300, [0.3]),
          ("tc", F32, 3, 5, 64, PINN, 5000, [0.3]), ("tc", F32, 2, 4, 64, RAYLEIGH, 3000, [0.3, -2.0]),
          ("tc", F32, 5, 5, 64, PINN, 2000, [0.3])]


@pytest.mark.parametrize("family,dtype,d,nl,H,kind,N,seed", LINEAR)
def test_seed_and_inv_n_are_linear(family, dtype, d, nl, H, kind, N, seed):
    """With a seed s and an arbitrary inv_n the gradient and dE are inv_n n sum_k s_k (those of seed e_k, inv_n = 1/n),
    the NULL seed is the all-ones seed, and the sums do not depend on either, bit for bit."""
    case = _case(dtype, d, nl, H, SIN, kind, ENV_POLY02, N, kind == PINN, seed=4)
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
    if kind == PINN:
        dE1 = float(units[0]["dE"][0])
        assert float(base["dE"][0]) == pytest.approx(dE1, rel=tol, abs=0)
        assert float(got["dE"][0]) == pytest.approx(inv_n * N * float(s[0]) * dE1, rel=tol, abs=0)


# ================================================================================================ (e) output contract
# family, dtype, d, n_linear, H, program, N
CONTRACT = [("simt", F64, 2, 3, 20, PINN, 300), ("simt", F32, 1, 4, 256, RAYLEIGH, 149), ("tc", F32, 3, 5, 64, PINN, 1000),
            ("tc", F32, 2, 4, 64, RAYLEIGH, 5000), ("tc", F32, 5, 5, 64, PINN, 500)]


@pytest.mark.parametrize("family,dtype,d,nl,H,kind,N", CONTRACT)
def test_residual_outputs_and_workspace_carry_no_state(family, dtype, d, nl, H, kind, N):
    """sums, grad and energy_grad are pure outputs and the workspace holds nothing across calls: with every byte of
    them NaN beforehand the results are bit-identical to a run on zeroed buffers, nothing past their ends is written,
    and grad = NULL with energy_grad set still gives the same dE and sums."""
    case = _case(dtype, d, nl, H, TANH, kind, ENV_POLY02, N, kind == PINN, seed=5)
    K = NQ[kind]
    with _path(family):
        clean = case.run(fill=0)
        dirty = case.run(fill=POISON)
        no_grad = case.run(fill=POISON, grad=False)
    assert clean["path"] == dirty["path"] == no_grad["path"] == (1 if family == "tc" else 0)
    assert clean["intact"] and dirty["intact"] and no_grad["intact"]
    for k, n in (("sums", K), ("grad", case.net.n_params), ("dE", 1)):
        assert torch.equal(_bytes(dirty[k], n), _bytes(clean[k], n)), k
    assert torch.equal(_bytes(no_grad["sums"], K), _bytes(clean["sums"], K))
    assert torch.equal(_bytes(no_grad["dE"], 1), _bytes(clean["dE"], 1))
    assert torch.isfinite(clean["grad"]).all() and torch.isfinite(clean["sums"]).all()


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
