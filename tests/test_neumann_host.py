"""CPU tests of the boundary-flux program (PDE_PROG_FLUX): its C ABI description, the Python descriptors, and the
float64 autograd specification the GPU tests compare the kernels against (tests/flux_oracle.py)."""
import ctypes as C
import math

import pytest
import torch

import pde_b200 as pb
from pde_b200 import _lib as L
from pde_b200.ops import ProgramSpec

from flux_oracle import flux_loss, manufactured_flux


def test_flux_program_is_one_quantity_of_order_one():
    lib = pb.load_library()
    assert L.PROG_FLUX == 5
    assert lib.pde_program_quantities(5) == 1 and lib.pde_program_order(5) == 1
    assert lib.pde_program_quantities(6) < 0 and lib.pde_program_order(6) < 0
    assert "pde_sample_faces_rhs" in L.EXPORTS


def test_program_faces_field_takes_the_reserved_slot():
    assert L.Program.faces.offset == 4 and L.Program.alpha.offset == 8
    assert C.sizeof(L.Program) == 56
    for m in (0b1, 0b100101, (1 << 10) - 1):
        assert ProgramSpec(L.PROG_FLUX, 2.0, faces=m).to_c().faces == m
    assert ProgramSpec(L.PROG_PINN).to_c().faces == 0          # every existing caller leaves it 0


def _masks(d):
    out = [1, 1 << (2 * d - 1), 3 << (2 * (d - 1)), (1 << 2 * d) - 1]
    if d == 2:
        out.append(0b1001)
    if d >= 3:
        out.append(0b100101)
    return out


@pytest.mark.parametrize("d", [1, 2, 3, 4, 5])
def test_oracle_known_answer_is_zero_for_the_manufactured_solution(d):
    """flux_loss with u* in place of the network and g from the closed form is 0 (float64); a wrong sign of the
    normal, a wrong block or a wrong axis would leave (k pi / L)^2-sized residuals."""
    L_box, per = 2.0, 37
    ks = [1 + (i % 3) for i in range(d)]
    gen = torch.Generator().manual_seed(d)
    u_star = lambda X: pb.poisson.exact_u_prod_sin(X, L_box, ks)
    for mask in _masks(d):
        faces = [k for k in range(2 * d) if mask >> k & 1]
        X = torch.rand(per * len(faces), d, dtype=torch.float64, generator=gen) * L_box
        for j, k in enumerate(faces):
            X[j * per:(j + 1) * per, k // 2] = L_box if k % 2 else 0.0
        g = manufactured_flux(X, mask, L_box, ks)
        assert float(g.abs().max()) > 0.1
        Xg = X.clone().requires_grad_(True)
        assert float(flux_loss(u_star, Xg, mask, g, L_box, "RB").detach()) <= 1e-12, mask
        # Robin: alpha du/dn + kappa u = alpha g + kappa u*
        kappa = 0.7
        g_r = 1.5 * g + kappa * u_star(X).reshape(-1)
        assert float(flux_loss(u_star, Xg, mask, g_r, L_box, "RB", alpha=1.5, kappa=kappa).detach()) <= 1e-12, mask
        # the other sign of the normal is not a solution
        assert float(flux_loss(u_star, Xg, mask, -g, L_box, "RB").detach()) > 1e-3


def test_neumann_drop_in_refuses_a_bad_face_mask():
    m = pb.poisson.SolutionNet(2, 8, 3, "RB").double()
    for bad in (0, 1 << 4, -1):
        with pytest.raises(ValueError):
            pb.poisson.boundary_loss_neumann(m, 2.0, 10, 2, "cpu", faces=bad)
