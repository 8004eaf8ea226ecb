"""CPU tests of the Ritz value program (PDE_PROG_RITZ_VALUE): its C ABI description, the Python descriptor, the refusals
of FusedTrainer's Ritz boundary term and mean constraint, and the float64 specification the GPU tests compare the kernels
against (tests/ritz_oracle.py)."""
import math

import pytest
import torch

import pde_b200 as pb
from pde_b200 import _lib as L
from pde_b200.ops import ProgramSpec

from ritz_oracle import boundary_energy, exact_mean, ritz_energy, ritz_value_loss


def test_ritz_value_program_is_one_quantity_of_order_zero():
    lib = pb.load_library()
    assert L.PROG_RITZ_VALUE == 7
    assert lib.pde_program_quantities(7) == 1 and lib.pde_program_order(7) == 0
    # kind 6 stays unassigned, kind 8 does not exist
    for kind in (6, 8):
        assert lib.pde_program_quantities(kind) < 0 and lib.pde_program_order(kind) < 0


def test_ritz_program_spec_fields():
    p = ProgramSpec(L.PROG_RITZ_VALUE, alpha=-1.0, beta_const=1.5).to_c()
    assert (p.kind, p.faces, p.alpha, p.beta_const, p.energy_const) == (7, 0, -1.0, 1.5, 0.0)
    assert p.f is None and p.beta is None and p.energy is None
    f = torch.zeros(4, dtype=torch.float64)
    p = ProgramSpec(kind=7, alpha=0.0, beta_const=0.25).to_c(f=f)
    assert p.kind == 7 and p.f == f.data_ptr() and p.alpha == 0.0 and p.beta_const == 0.25


def _rb(dim=2):
    return pb.poisson.SolutionNet(dim, 8, 3, "RB").double()


def _no_launch(monkeypatch):
    """Any sampler or residual launch fails the test: the refusals come first."""
    def boom(*a, **k):
        raise AssertionError("launched before refusing")
    monkeypatch.setattr(pb.train, "sample_points_rhs", boom)
    monkeypatch.setattr(pb.train, "sample_faces_rhs", boom)
    monkeypatch.setattr(pb.train, "_residual_row", boom)


def test_trainer_refuses_ritz_form_with_pinn_or_without_faces(monkeypatch):
    _no_launch(monkeypatch)
    with pytest.raises(ValueError, match="DRM"):
        pb.train.FusedTrainer(_rb(), 2.0, [1, 1], method="PINN", neumann_faces=0b1111, neumann_form="ritz", graph=False)
    with pytest.raises(ValueError, match="neumann_faces"):
        pb.train.FusedTrainer(_rb(), 2.0, [1, 1], method="DRM", neumann_form="ritz", graph=False)
    with pytest.raises(ValueError):
        pb.train.FusedTrainer(_rb(), 2.0, [1, 1], method="DRM", neumann_faces=0b1111, neumann_form="natural", graph=False)


def test_trainer_refuses_weight_neumann_with_ritz_form(monkeypatch):
    _no_launch(monkeypatch)
    with pytest.raises(ValueError, match="weight_neumann"):
        pb.train.FusedTrainer(_rb(), 2.0, [1, 1], method="DRM", neumann_faces=0b1111, neumann_form="ritz",
                              weight_neumann=2.0, graph=False)


def test_trainer_refuses_mean_value_with_group(monkeypatch):
    _no_launch(monkeypatch)
    with pytest.raises(NotImplementedError, match="global mean"):
        pb.train.FusedTrainer(_rb(), 2.0, [1, 1], method="DRM", neumann_faces=0b1111, mean_value=True,
                              group=object(), graph=False)


def test_oracle_value_program_terms():
    torch.manual_seed(0)
    X = torch.rand(50, 3, dtype=torch.float64) * 2.0
    u = lambda Z: Z.sum(dim=1, keepdim=True) - 1.0
    g = torch.rand(50, dtype=torch.float64)
    uv = u(X).reshape(-1)
    assert torch.isclose(ritz_value_loss(u, X, None, 2.0, "RB", alpha=-1.0), uv.mean())
    assert torch.isclose(ritz_value_loss(u, X, g, 2.0, "RB", kappa=1.5), (0.75 * uv * uv - g * uv).mean())
    beta = torch.rand(50, dtype=torch.float64)
    assert torch.isclose(ritz_value_loss(u, X, None, 2.0, "RB", kappa=beta, alpha=0.3), (0.5 * beta * uv * uv - 0.3 * uv).mean())
    assert torch.isclose(boundary_energy(u, X, 0b100101, g, 2.0, "RB", 1.5),
                         1.5 * (0.75 * uv * uv - g * uv).mean())


def _midpoints(m, L_box):
    return (torch.arange(m, dtype=torch.float64) + 0.5) * (L_box / m)


@pytest.mark.parametrize("kappa", [0.0, 1.5])
def test_manufactured_solution_is_stationary_for_the_ritz_functional(kappa):
    """On a midpoint-rule grid of [0, L]^2 the first variation of E[u] / |Omega| at u = u* in the direction of a v that
    does not vanish on the boundary is ~0 when g = du*/dn + kappa u* on every face (non-integer ks, so that u* is not 0
    on the hi faces), and it is not 0 with a wrong boundary weight or without the kappa u* part of g."""
    L_box, ks, m = 2.0, [0.75, 1.3], 400
    t = _midpoints(m, L_box)
    X = torch.cartesian_prod(t, t).requires_grad_(True)
    f = pb.poisson.rhs_f_for_u_sin(X.detach(), L_box, ks)
    mask = 0b1111
    blocks = []
    for k in range(4):
        B = torch.stack([t, t], dim=1)
        B[:, k // 2] = L_box if k % 2 else 0.0
        blocks.append(B)
    Xb = torch.cat(blocks)
    from flux_oracle import manufactured_flux
    u_star = lambda Z: pb.poisson.exact_u_prod_sin(Z, L_box, ks)
    g_right = manufactured_flux(Xb, mask, L_box, ks) + kappa * u_star(Xb).reshape(-1)
    v = lambda Z: 1.0 + Z[:, 0:1] + 0.5 * Z[:, 1:2] ** 2

    def variation(g, scale=1.0):
        eps = torch.zeros((), dtype=torch.float64, requires_grad=True)
        net = lambda Z: u_star(Z) + eps * v(Z)
        e_in = ritz_energy(net, X, f, Xb, mask, g, L_box, "RB", kappa)
        e_b = boundary_energy(net, Xb, mask, g, L_box, "RB", kappa)
        (d,) = torch.autograd.grad(e_in + (scale - 1.0) * e_b, eps)
        return float(d)

    assert abs(variation(g_right)) <= 2e-4
    assert abs(variation(g_right, scale=L_box)) > 1e-2           # the boundary integral not divided by L
    if kappa:
        assert abs(variation(manufactured_flux(Xb, mask, L_box, ks))) > 1e-2


def test_exact_mean_of_the_manufactured_solution():
    L_box, ks, m = 2.0, [1.0, 2.0, 0.75], 60
    t = _midpoints(m, L_box)
    X = torch.cartesian_prod(t, t, t)
    got = float(pb.poisson.exact_u_prod_sin(X, L_box, ks).mean())
    assert abs(got - exact_mean(L_box, ks)) <= 1e-3 * max(abs(exact_mean(L_box, ks)), 1e-3)
    assert exact_mean(L_box, [2.0]) == pytest.approx(0.0, abs=1e-15) and exact_mean(L_box, [1.0]) == pytest.approx(2 / math.pi)
