"""GPU parity of both kernel families on boxes of every size (run with -m gpu on a B200).

The tensor-core kernel splits every GEMM operand into two fp16 parts.  The derivative channels of its jets scale with the
first-layer weights W0 (the Laplacian with W0^2), and a network trained on a box of side L has W0 ~ 1 / L, so the box
size decides how close those operands come to fp16's subnormal range.  Here W0 of a seeded network is multiplied by
p = 2^round(log2(2 / L)) and the points are drawn in a box of side L, so that W0 x + b covers the same range at every L in
{1/32, 1/4, 2, 20, 60, 200, 2000}.  The program coefficients that multiply derivatives carry the matching powers of 1 / p
(exact), so that every term of every residual stays O(1) and the loss depends on the derivative channels at every L.

References: oracle/jets_numpy and tests/flux_oracle.py in float64, and the float64 generic kernel at 2^20 points.
Bar: 1e-5 relative in fp32, raised only by the conftest.py rule (twice the reference algorithm's own float32 error)."""
import math

import numpy as np
import pytest
import torch

from conftest import assert_grads_close, grads_err
from test_gpu_tc import _grads, _rand_net, _reference_fp32_error_rayleigh, _seq

pytestmark = pytest.mark.gpu
TOL = 1e-5
BOXES = [1 / 32, 1 / 4, 2.0, 20.0, 60.0, 200.0, 2000.0]
POLY_BOXES = [L for L in BOXES if L <= 20]   # the POLY envelope grows like (L / 2)^(2 d)
FAMILY = {"tc": "tcgen05", "simt": "simt_fma"}


def _f32(a):
    """values the float32 kernels see exactly"""
    return np.asarray(a, dtype=np.float64).astype(np.float32).astype(np.float64)


def _p(L):
    """the power of two nearest to 2 / L"""
    return 2.0 ** round(math.log2(2.0 / L))


def _box_net(seed, d, w, depth, L):
    rng = np.random.default_rng(seed)
    Ws, bs = _rand_net(rng, d, w, depth)
    Ws[0] = Ws[0] * _p(L)
    return rng, Ws, bs


def _points(rng, N, d, lo, L):
    return _f32(lo + L * rng.uniform(0.0, 1.0, (N, d)))


def _env(kind, lo, hi, nodes=None):
    return {"kind": kind, "lo": lo, "hi": hi, "nodes": nodes}


def _run_program(Ws, bs, X, act, prog, env, path, alpha, f=None, beta=None, E=0.0):
    """(kernel loss, kernel grads, oracle loss, oracle grads) of one residual program through ops.residual_means."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import EnvelopeSpec, ProgramSpec, residual_means
    from oracle import jets_numpy as O
    N, d = X.shape
    A = O.SIN if act == "sin" else O.TANH
    espec = EnvelopeSpec(env["kind"], env["lo"], env["hi"], env["nodes"] or [])
    net, lin = _seq(Ws, bs, act)
    dev = lambda a: None if a is None else torch.tensor(a, dtype=torch.float32, device="cuda")
    Xg = dev(X)
    with pb.ops.kernel_path(path):
        if prog == "pinn":
            want, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, A, env, alpha, beta, E, f=f)
            loss = residual_means(net, Xg, ProgramSpec(L.PROG_PINN, alpha, 0.0, E), espec, f=dev(f), beta=dev(beta))[0]
        elif prog == "drm":
            def program(U):   # q = alpha |grad u|^2 - f u, the kernel's Deep Ritz program with a free alpha
                u, g = U[:, 0:1], U[:, 1:1 + d]
                Ubar = np.zeros_like(U)
                Ubar[:, 0:1] = -f
                Ubar[:, 1:1 + d] = 2.0 * alpha * g
                return float((alpha * np.sum(g * g, axis=1, keepdims=True) - f * u).mean()), Ubar / N, None
            want, gWs, gbs, _ = O._loss_and_grads(Ws, bs, X, A, 1, env, program)
            loss = residual_means(net, Xg, ProgramSpec(L.PROG_DRM, alpha), espec, f=dev(f))[0]
        else:
            want, gWs, gbs, _ = O.rayleigh_loss(Ws, bs, X, A, env, alpha, beta)
            m = residual_means(net, Xg, ProgramSpec(L.PROG_RAYLEIGH, alpha), espec, beta=dev(beta))
            loss = m[0] / m[1]
        assert pb.ops.last_kernel_path() == FAMILY[path]
        loss.backward()
    return float(loss.detach()), _grads(lin), want, (gWs, gbs)


def _assert_close(got, ggot, want, gwant, bar, what):
    # losses with cancelling terms (Deep Ritz) are compared on the scale of their terms, as in test_gpu_tc
    assert abs(got - want) <= bar * max(abs(want), 1e-2), (what, got, want)
    assert_grads_close(ggot, gwant, bar, what)


PINN_CASES = [(d, act, env, L) for d in (1, 3) for act in ("sin", "tanh")
              for env, boxes in (("none", BOXES), ("poly", POLY_BOXES)) for L in boxes]


@pytest.mark.parametrize("path", ["tc", "simt"])
@pytest.mark.parametrize("d,act,env_kind,L", PINN_CASES)
def test_pinn_across_box_sizes(d, act, env_kind, L, path):
    """alpha Lap u + (beta - E) u - f with alpha = -1 / p^2, per-point beta; no envelope, or POLY on [0, L].  With the
    envelope, u is of the size of B ~ (L / 2)^(2 d), and so is f: a residual that is -f alone on a small box would
    make the gradient a sum of random-sign terms that cancel, whatever the kernel."""
    from oracle import jets_numpy as O
    rng, Ws, bs = _box_net(10 * d + (act == "tanh"), d, 64, 5, L)
    N = 2000
    X = _points(rng, N, d, 0.0, L)
    f = _f32(rng.normal(size=(N, 1)) * ((L / 2) ** (2 * d) if env_kind == "poly" else 1.0))
    beta = _f32(rng.uniform(0.5, 1.5, (N, 1)))
    env = _env(O.ENV_POLY if env_kind == "poly" else O.ENV_NONE, 0.0, L)
    got, gg, want, gw = _run_program(Ws, bs, X, act, "pinn", env, path, -1.0 / _p(L) ** 2, f=f, beta=beta, E=0.3)
    _assert_close(got, gg, want, gw, TOL, f"pinn d{d} {act} {env_kind} L={L} {path}")


@pytest.mark.parametrize("L", BOXES)
def test_tc_deep_ritz_across_box_sizes(L):
    from oracle import jets_numpy as O
    rng, Ws, bs = _box_net(20, 2, 64, 5, L)
    N = 2000
    X = _points(rng, N, 2, 0.0, L)
    f = _f32(rng.normal(size=(N, 1)))
    got, gg, want, gw = _run_program(Ws, bs, X, "sin", "drm", _env(O.ENV_NONE, 0.0, L), "tc", 0.5 / _p(L) ** 2, f=f)
    _assert_close(got, gg, want, gw, TOL, f"drm L={L}")


@pytest.mark.parametrize("L", BOXES)
def test_tc_rayleigh_across_box_sizes(L):
    """mean(a |grad u|^2 + beta u^2) / mean(u^2), a = 1 / (2 p^2), per-point beta, POLY envelope on [0, L] (the
    envelope of the reference algorithm whose float32 error sets the bar)."""
    from oracle import jets_numpy as O
    rng, Ws, bs = _box_net(30, 2, 50, 5, L)
    N = 1500
    X = _points(rng, N, 2, 0.0, L)
    beta = _f32(rng.uniform(0.5, 1.5, (N, 1)))
    a = 0.5 / _p(L) ** 2
    got, gg, want, gw = _run_program(Ws, bs, X, "sin", "rayleigh", _env(O.ENV_POLY, 0.0, L), "tc", a, beta=beta)
    bar = max(TOL, 2.0 * _reference_fp32_error_rayleigh(Ws, bs, X, beta, "sin", a, L))
    _assert_close(got, gg, want, gw, bar, f"rayleigh L={L}")


@pytest.mark.parametrize("L", BOXES)
def test_tc_expwin_with_forced_nodes_across_box_sizes(L):
    """The Schroedinger shape: EXPWIN window on [-L/2, L/2] with two forced nodes on x_0, -1/(2 p^2) Lap u + (V - E) u."""
    from oracle import jets_numpy as O
    rng, Ws, bs = _box_net(40, 2, 64, 5, L)
    N = 2000
    X = _points(rng, N, 2, -L / 2, L)
    V = _f32(rng.uniform(0.5, 1.5, (N, 1)))
    env = _env(O.ENV_EXPWIN, -L / 2, L / 2, [[-L / 8, L / 4], []])
    got, gg, want, gw = _run_program(Ws, bs, X, "sin", "pinn", env, "tc", -0.5 / _p(L) ** 2, beta=V, E=0.3)
    _assert_close(got, gg, want, gw, TOL, f"expwin L={L}")


@pytest.mark.parametrize("path", ["tc", "simt"])
@pytest.mark.parametrize("L", [1 / 32, 60.0])
def test_pinn_5d_across_box_sizes(L, path):
    """Seven jet channels: on the tensor-core kernel the two dimension-split passes around the pointwise residual kernel."""
    from oracle import jets_numpy as O
    rng, Ws, bs = _box_net(50, 5, 64, 5, L)
    N = 3000
    X = _points(rng, N, 5, 0.0, L)
    f = _f32(rng.normal(size=(N, 1)))
    beta = _f32(rng.uniform(0.5, 1.5, (N, 1)))
    got, gg, want, gw = _run_program(Ws, bs, X, "sin", "pinn", _env(O.ENV_NONE, 0.0, L), path, -1.0 / _p(L) ** 2,
                                     f=f, beta=beta, E=0.3)
    _assert_close(got, gg, want, gw, TOL, f"5-D pinn L={L} {path}")


@pytest.mark.parametrize("path", ["tc", "simt"])
@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("L", [1 / 32, 60.0])
def test_jets_forward_backward_across_box_sizes(L, order, path):
    """pde_jets_forward / pde_jets_backward (the WAN path): each channel block of the jets against its own largest entry,
    and the reverse sweep with derivative cotangents of size 1 / p, so that every channel reaches the gradient."""
    import pde_b200 as pb
    from oracle import jets_numpy as O
    d = 3
    rng, Ws, bs = _box_net(60 + order, d, 64, 5, L)
    N = 2000
    X = _points(rng, N, d, 0.0, L)
    Jbar = _f32(rng.normal(size=(N, 1 + order * d)))
    Jbar[:, 1:] /= _p(L)
    J, cache = O.mlp_jets_forward(Ws, bs, X, O.SIN, order)
    gWs, gbs = O.mlp_jets_backward(Ws, bs, cache, Jbar)
    net, lin = _seq(Ws, bs, "sin")
    with pb.ops.kernel_path(path):
        Jg = pb.mlp_jets(net, torch.tensor(X, dtype=torch.float32, device="cuda"), order)
        assert pb.ops.last_kernel_path() == FAMILY[path]
        Jg.backward(torch.tensor(Jbar, dtype=torch.float32, device="cuda"))
        assert pb.ops.last_kernel_path() == FAMILY[path]
    Jn = Jg.detach().double().cpu().numpy()
    # the bias gradients of random-sign cotangents cancel (order 0 most): the bar follows the conftest.py rule, twice the
    # float32 error of the same algorithm (the oracle run in float32), worst of this case and four inputs one ulp away
    gen = np.random.default_rng(1)
    e32 = 0.0
    for k in range(5):
        jit = (lambda t: t * (1.0 + gen.uniform(-1, 1, np.shape(t)) * 2.0 ** -24)) if k else (lambda t: t)
        W, b, Xj, Jbj = [jit(v) for v in Ws], [jit(v) for v in bs], jit(X), jit(Jbar)
        run = lambda dt: O.mlp_jets_backward([v.astype(dt) for v in W], [v.astype(dt) for v in b],
                                             O.mlp_jets_forward([v.astype(dt) for v in W], [v.astype(dt) for v in b], Xj.astype(dt),
                                                                O.SIN, order)[1], Jbj.astype(dt))
        e32 = max(e32, grads_err(run(np.float32), run(np.float64))[0])
    bar = max(TOL, 2.0 * e32)
    for blk in ([0], list(range(1, 1 + order * d))):
        if blk:
            err = np.max(np.abs(Jn[:, blk] - J[:, blk])) / np.max(np.abs(J[:, blk]))
            assert err <= 5 * TOL, (blk, err)
    assert_grads_close(_grads(lin), (gWs, gbs), bar, f"jets order {order} L={L} {path}")


@pytest.mark.parametrize("L", BOXES)
def test_tc_flux_program_across_box_sizes(L):
    """alpha n.grad u + kappa u - g on all six faces of [0, L]^3, alpha = 1 / p, per-point kappa."""
    from test_gpu_neumann import _e32, _kernel, _net, _oracle
    rng = np.random.default_rng(80)
    net = _net(rng, 3, 32, 4, "sin")
    with torch.no_grad():
        net[0].weight.mul_(_p(L))
    mask, per = 0b111111, 200
    X = _points(rng, 6 * per, 3, 0.0, L)
    for k in range(6):
        X[k * per:(k + 1) * per, k // 2] = L if k % 2 else 0.0
    g = _f32(rng.normal(size=6 * per))
    kappa = _f32(rng.uniform(0.5, 1.5, 6 * per))
    alpha = 1.0 / _p(L)
    want, wgrads = _oracle(net, X, mask, g, "RB", alpha, kappa)
    bar = max(TOL, 2.0 * _e32(net, X, mask, g, "RB", alpha, kappa))
    got, ggrads, fam = _kernel(net, X, mask, g, "RB", alpha, kappa, torch.float32, "tc")
    assert fam == "tcgen05"
    assert abs(got - want) <= bar * max(abs(want), 1e-3), (got, want, bar)
    e, where = grads_err(ggrads, wgrads)
    assert e <= bar, (where, e, bar)


def test_tc_large_batch_on_a_large_box_against_fp64_generic_kernel():
    """2^20 points on [0, 200)^3 (several tiles per CTA, each with its own adjoint scale): the fp32 tensor-core kernel
    against the generic kernel in fp64 on the same points."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import NO_ENVELOPE, ProgramSpec, residual_means
    box = 200.0
    _, Ws, bs = _box_net(90, 3, 64, 5, box)
    n32, lin32 = _seq(Ws, bs, "sin")
    n64, lin64 = _seq(Ws, bs, "sin", torch.float64)
    N = 1 << 20
    gen = torch.Generator(device="cuda").manual_seed(90)
    X = torch.rand(N, 3, device="cuda", generator=gen) * box
    f = torch.randn(N, device="cuda", generator=gen)
    spec = ProgramSpec(L.PROG_PINN, -1.0 / _p(box) ** 2)
    with pb.ops.kernel_path("tc"):
        l32 = residual_means(n32, X, spec, NO_ENVELOPE, f=f)[0]
        assert pb.ops.last_kernel_path() == "tcgen05"
        l32.backward()
    with pb.ops.kernel_path("simt"):
        l64 = residual_means(n64, X.double(), spec, NO_ENVELOPE, f=f.double())[0]
        l64.backward()
    assert abs(l32.item() - l64.item()) <= TOL * abs(l64.item())
    assert_grads_close(_grads(lin32), _grads(lin64), TOL, "2^20 points, L = 200")


def test_tc_sin_beyond_2_15_against_oracle():
    """First-layer pre-activations past 2^15, where the tensor-core kernel leaves its Cody-Waite sin / cos for the
    library's: 1-D points on [0, 40000) in increasing order, so that the first tiles stay below 2^15 and the last ones
    cross it.  W0 = k / 8 (|k| <= 8), b0 = m / 4 and integer x make every W0 x + b0 exact in fp32, so the float64 oracle
    sees the kernel's arguments."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import NO_ENVELOPE, ProgramSpec, residual_means
    from oracle import jets_numpy as O
    rng = np.random.default_rng(12)
    w, N = 32, 64 * 64
    Ws, bs = _rand_net(rng, 1, w, 4)
    k = rng.integers(1, 9, w) * rng.choice([-1, 1], w)
    k[::5] = 8 * np.sign(k[::5])
    Ws[0] = (k / 8.0).reshape(w, 1)
    bs[0] = rng.integers(-8, 9, w) / 4.0
    X = np.sort(rng.integers(0, 40000, N)).astype(np.float64).reshape(N, 1)
    zmax = np.abs(X @ Ws[0].T + bs[0]).reshape(N // 64, -1).max(axis=1)
    assert (zmax > 2 ** 15).any() and (zmax < 2 ** 15).any()
    net, lin = _seq(Ws, bs, "sin")
    Xg = torch.tensor(X, dtype=torch.float32, device="cuda")
    J = O.mlp_jets_forward(Ws, bs, X, O.SIN, 1)[0]
    with pb.ops.kernel_path("tc"):
        Jg = pb.mlp_jets(net, Xg, 1).detach().double().cpu().numpy()
        assert pb.ops.last_kernel_path() == "tcgen05"
    for c in range(2):
        err = np.max(np.abs(Jg[:, c] - J[:, c])) / np.max(np.abs(J[:, c]))
        assert err <= 5 * TOL, (c, err)
    f = _f32(rng.normal(size=(N, 1)))
    beta = _f32(rng.uniform(0.5, 1.5, (N, 1)))
    want, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, O.SIN, _env(O.ENV_NONE, 0.0, 40000.0), -1.0, beta, 0.3, f=f)
    net.zero_grad()
    dev = lambda a: torch.tensor(a, dtype=torch.float32, device="cuda")
    with pb.ops.kernel_path("tc"):
        loss = residual_means(net, Xg, ProgramSpec(L.PROG_PINN, -1.0, 0.0, 0.3), NO_ENVELOPE, f=dev(f), beta=dev(beta))[0]
        assert pb.ops.last_kernel_path() == "tcgen05"
        loss.backward()
    _assert_close(float(loss.detach()), _grads(lin), want, (gWs, gbs), TOL, "sin past 2^15")
