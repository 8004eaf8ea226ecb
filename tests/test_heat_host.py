"""CPU tests of the parabolic program (PDE_PROG_PARABOLIC): its C ABI description, the refusals the library answers
before it enqueues anything, the float64 specification the GPU tests compare the kernels against (tests/heat_oracle.py)
and the argument checks of pde_b200.heat."""
import ctypes as C

import pytest
import torch

import pde_b200 as pb
from pde_b200 import _lib as L

from heat_oracle import parabolic_loss, parabolic_residual

DUMMY = 0x100000   # never dereferenced: every call below is refused before anything is enqueued


def test_parabolic_program_is_one_quantity_of_order_two():
    lib = pb.load_library()
    assert L.PROG_PARABOLIC == 9
    assert lib.pde_program_quantities(9) == 1 and lib.pde_program_order(9) == 2
    for kind in (6, 8):   # still unassigned
        assert lib.pde_program_quantities(kind) < 0 and lib.pde_program_order(kind) < 0


def test_face_masks_put_time_last():
    assert pb.heat.spatial_faces(2) == 0b11 and pb.heat.initial_face(2) == 0b100
    assert pb.heat.spatial_faces(4) == 0b111111 and pb.heat.initial_face(4) == 1 << 6
    for d in range(2, 6):
        assert pb.heat.spatial_faces(d) & pb.heat.initial_face(d) == 0
        assert (pb.heat.spatial_faces(d) | pb.heat.initial_face(d)) < pb.train.all_faces(d)


def _c_net(dim):
    n = L.Net()
    n.dtype, n.dim, n.n_linear, n.activation = L.F32, dim, 3, L.ACT_SIN
    for i, w in enumerate([dim, 8, 8, 1]):
        n.widths[i] = w
    for l in range(3):
        n.W[l] = n.b[l] = DUMMY
    return n


def _refusals():
    """(dim, envelope or None) of every refused call."""
    out = [(1, None)]
    env = L.Envelope()
    env.kind, env.lo, env.hi = L.ENV_POLY, 0.0, 1.0
    out.append((3, env))
    env = L.Envelope()
    env.kind, env.lo, env.hi = L.ENV_EXPWIN, 0.0, 1.0
    out.append((3, env))
    for i in (0, 2):   # no envelope kind, but forced nodes on a spatial axis or on time
        env = L.Envelope()
        env.kind = L.ENV_NONE
        env.n_nodes[i] = 1
        out.append((3, env))
    return out


@pytest.mark.parametrize("case", range(5))
def test_library_refuses_before_enqueueing(case):
    lib = pb.load_library()
    dim, env = _refusals()[case]
    net = _c_net(dim)
    prog = L.Program()
    prog.kind, prog.alpha = L.PROG_PARABOLIC, -1.0
    envp = None if env is None else C.byref(env)
    rc = lib.pde_residual_loss_grad(C.byref(net), envp, C.byref(prog), DUMMY, 4096, None, 1.0 / 4096, DUMMY, DUMMY,
                                    None, DUMMY, 1 << 30, None)
    assert rc == -1, rc
    peers = L.Peers()
    peers.rank, peers.world = 0, 2
    peers.base[0] = peers.base[1] = DUMMY
    rc = lib.pde_residual_loss_grad_exchange(C.byref(net), envp, C.byref(prog), DUMMY, 4096, None, 1.0 / 4096, DUMMY,
                                             DUMMY, 1 << 30, C.byref(peers), 1 << 20, DUMMY, None)
    assert rc == -1, rc


def _loss(*a, **k):
    return float(parabolic_loss(*a, **k).detach())


@pytest.mark.parametrize("d", [2, 3, 4, 5])
def test_oracle_vanishes_on_the_heat_solution(d):
    torch.manual_seed(d)
    L_box, kappa = 1.5, 0.7
    ks = [1, 2, 1, 3][:d - 1]
    X = (torch.rand(64, d, dtype=torch.float64) * L_box).requires_grad_(True)
    u = lambda Z: pb.heat.exact_u_heat(Z, L_box, ks, kappa)
    assert _loss(u, X, None, alpha=-kappa) <= 1e-12
    # the wrong sign of alpha (a backward heat equation) leaves 2 u_t
    assert _loss(u, X, None, alpha=kappa) > 1e-2
    # beta, E and f enter as in the PINN program
    f = 0.3 * u(X.detach()).reshape(-1)
    assert _loss(u, X, f, alpha=-kappa, beta=0.5, E=0.2) <= 1e-12


def test_oracle_residual_terms():
    """r = u_t + alpha Lap_x u + (beta - E) u - f on a polynomial with known derivatives, time last."""
    X = torch.tensor([[0.5, -1.0, 2.0], [1.5, 0.25, -0.5]], dtype=torch.float64, requires_grad=True)
    u = lambda Z: (Z[:, 0:1] ** 2 + 3 * Z[:, 1:2] ** 2 * Z[:, 2:3] + Z[:, 2:3] ** 3)
    x0, x1, t = X.detach()[:, 0:1], X.detach()[:, 1:2], X.detach()[:, 2:3]
    ut = 3 * x1 ** 2 + 3 * t ** 2
    lap = 2 + 6 * t   # the t^3 term's second t-derivative stays out
    f = torch.tensor([0.1, -0.2], dtype=torch.float64)
    want = ut + 0.4 * lap + (1.5 - 0.5) * u(X.detach()) - f.reshape(-1, 1)
    got = parabolic_residual(u, X, f, alpha=0.4, beta=1.5, E=0.5)
    assert torch.allclose(got, want, rtol=1e-14, atol=1e-13)


def test_exact_u_heat_initial_and_boundary_values():
    ks, L_box, kappa = [1, 2], 2.0, 0.3
    X = torch.rand(32, 3, dtype=torch.float64) * L_box
    X0 = X.clone()
    X0[:, 2] = 0.0
    init = torch.sin(torch.pi * X0[:, 0:1] / L_box) * torch.sin(2 * torch.pi * X0[:, 1:2] / L_box)
    assert torch.allclose(pb.heat.exact_u_heat(X0, L_box, ks, kappa), init, atol=1e-15)
    Xb = X.clone()
    Xb[:, 1] = L_box
    assert float(pb.heat.exact_u_heat(Xb, L_box, ks, kappa).abs().max()) <= 1e-14
    with pytest.raises(ValueError):
        pb.heat.exact_u_heat(X, L_box, [1], kappa)


def test_drop_in_refuses_before_launching(monkeypatch):
    def boom(*a, **k):
        raise AssertionError("launched before refusing")
    monkeypatch.setattr(pb.heat, "residual_mean", boom)
    X = torch.rand(16, 3)
    with pytest.raises(ValueError, match="FBC"):
        pb.heat.heat_residual_loss(pb.poisson.SolutionNet(3, 8, 3, "FBC"), X)
    with pytest.raises(ValueError, match="d >= 2"):
        pb.heat.heat_residual_loss(pb.poisson.SolutionNet(1, 8, 3, "RB"), torch.rand(16, 1))
    with pytest.raises(ValueError, match="d >= 2"):
        pb.heat.heat_residual_loss(pb.poisson.SolutionNet(1, 8, 3, "RB"), torch.rand(16))
