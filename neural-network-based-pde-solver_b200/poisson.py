"""Drop-in for the loss-function API of ``Poisson_Equations/Poisson_ND.py``.

Same names, argument order and return arity as the reference (file:line cited per function);
the loss step itself runs in the fused CUDA kernels.  The functions accept the reference's own
``SolutionNet`` / ``CriticNet`` objects as well as the classes defined here (identical layout:
``.net`` is an ``nn.Sequential`` with Linear at even indices, ``.bc_mode`` selects the envelope).
Extra keyword-only arguments ``group`` / ``n_global`` give exact data parallelism over points.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import _lib
from .ops import (NO_ENVELOPE, EnvelopeSpec, ProgramSpec, WanSpec, mlp_jets, residual_mean, residual_means, wan_means,
                  wan_scalar_losses)


class Sin(nn.Module):
    """sin activation (Poisson_ND.py:8-9)."""

    def forward(self, x):
        return torch.sin(x)


def _stack(in_f, width, depth):
    layers = []
    for _ in range(depth - 1):
        layers += [nn.Linear(in_f, width), Sin()]
        in_f = width
    layers += [nn.Linear(in_f, 1)]
    return nn.Sequential(*layers)


class SolutionNet(nn.Module):
    """u-network with optional hard Dirichlet envelope (Poisson_ND.py:11-33)."""

    def __init__(self, dim, width=64, depth=5, bc_mode='FBC'):
        super().__init__()
        self.dim, self.bc_mode = dim, bc_mode
        self.net = _stack(dim, width, depth)

    def forward(self, X, L=2.0):
        u = self.net(X)
        if self.bc_mode == 'FBC':
            return torch.prod(X * (L - X), dim=1, keepdim=True) * u
        if self.bc_mode == 'RB':
            return u
        raise ValueError("bc_mode must be 'FBC' or 'RB'")


class CriticNet(nn.Module):
    """adversarial test network v (Poisson_ND.py:35-46)."""

    def __init__(self, dim, width=64, depth=3):
        super().__init__()
        self.net = _stack(dim, width, depth)

    def forward(self, X):
        return self.net(X)


def exact_u_prod_sin(X, L, ks):
    """u*(x) = prod_i sin(k_i pi x_i / L)   (Poisson_ND.py:49-52)."""
    u = torch.ones(X.shape[0], 1, dtype=X.dtype, device=X.device)
    for i, k in enumerate(ks):
        u = u * torch.sin(k * math.pi * X[:, i:i + 1] / L)
    return u


def rhs_f_for_u_sin(X, L, ks):
    """f = (sum_i (k_i pi / L)^2) u*   (Poisson_ND.py:54-58)."""
    s = sum((k * math.pi / L) ** 2 for k in ks)
    return s * exact_u_prod_sin(X, L, ks)


def _envelope(model, L):
    mode = getattr(model, "bc_mode", 'RB')
    if mode == 'FBC':
        return EnvelopeSpec(_lib.ENV_POLY, 0.0, float(L))
    if mode == 'RB':
        return NO_ENVELOPE
    raise ValueError("bc_mode must be 'FBC' or 'RB'")





def pinn_residual_loss(model, X_in, f_in, L, *, group=None, n_global=None):
    """mean((-Lap u - f)^2)   (Poisson_ND.py:91-96)."""
    return residual_mean(model, X_in, ProgramSpec(_lib.PROG_PINN, alpha=-1.0), _envelope(model, L), f=f_in,
                         group=group, n_global=n_global)


def drm_energy_loss(model, X_in, f_in, L, *, group=None, n_global=None):
    """mean(1/2 |grad u|^2 - f u)   (Poisson_ND.py:98-103)."""
    return residual_mean(model, X_in, ProgramSpec(_lib.PROG_DRM, alpha=0.5), _envelope(model, L), f=f_in,
                         group=group, n_global=n_global)


def wan_losses(u_model, v_model, X, f_vals, L, eps=1e-8, v_reg_weight=0.0, *, group=None, n_global=None,
               u_jets=None, v_jets=None):
    """(loss_pde_u, loss_v, weak_residual, phi_norm)   (Poisson_ND.py:105-128)."""
    assert X.requires_grad, "X must require_grad=True"
    m = wan_means(u_model, v_model, X, WanSpec(alpha=1.0, w_lo=0.0, w_hi=float(L)), env_u=_envelope(u_model, L),
                  env_v=NO_ENVELOPE, f=f_vals, group=group, n_global=n_global, u_jets=u_jets, v_jets=v_jets)
    loss_pde_u, loss_v, _, _ = wan_scalar_losses(m, kind=0, eps_pde=eps, eps_log=eps, reg=v_reg_weight)
    return loss_pde_u, loss_v, m[0].detach(), m[1].detach()


def boundary_loss_dirichlet(model, L, N_b_per_face, dim, device, *, group=None):
    """mean over the 2d faces of mean(u(face)^2), fresh uniform face samples   (Poisson_ND.py:130-141)."""
    dtype = next(model.parameters()).dtype
    losses = []
    for i in range(dim):
        for at_L in (False, True):
            X = torch.rand(N_b_per_face, dim, device=device, dtype=dtype) * L
            X[:, i] = L if at_L else 0.0
            # (with group, residual_mean counts N_b_per_face points on every rank)
            losses.append(residual_mean(model, X, ProgramSpec(_lib.PROG_MSE), _envelope(model, L), group=group))
    return sum(losses) / len(losses)


def boundary_loss_neumann(model, L, N_b_per_face, dim, device, g=None, faces=None, *, group=None):
    """mean over the selected faces of mean((du/dn - g)^2), fresh uniform face samples: the Neumann counterpart of
    boundary_loss_dirichlet (Poisson_ND.py:130-141, same torch.rand face draws), one fused launch for all faces.

    ``faces``: face mask, face k = (coordinate k // 2, side k % 2: 0 or L), default every face; ``g``: None (zero flux)
    or a callable g(X) -> (N,) giving the prescribed outward normal derivative.  A Robin condition
    alpha du/dn + kappa u = g is ``ops.residual_mean`` with ``ProgramSpec(PROG_FLUX, alpha, beta_const=kappa,
    faces=mask)`` on the same blocked points."""
    dtype = next(model.parameters()).dtype
    mask = (1 << 2 * dim) - 1 if faces is None else int(faces)
    if not 0 < mask < 1 << 2 * dim:
        raise ValueError(f"faces must be a face mask in 1 .. {(1 << 2 * dim) - 1}")
    blocks = []
    for i in range(dim):
        for at_L in (False, True):
            if mask >> (2 * i + int(at_L)) & 1:
                X = torch.rand(N_b_per_face, dim, device=device, dtype=dtype) * L
                X[:, i] = L if at_L else 0.0
                blocks.append(X)
    X = torch.cat(blocks)
    gv = None if g is None else g(X).reshape(-1)
    # (with group, residual_mean counts the points of this rank on every rank)
    return residual_mean(model, X, ProgramSpec(_lib.PROG_FLUX, faces=mask), _envelope(model, L), f=gv, group=group)


def data_loss(model, X_data, u_data, L, *, group=None, n_global=None):
    """mean((u(X_data) - u_data)^2)   (Poisson_ND.py:230-232)."""
    return residual_mean(model, X_data, ProgramSpec(_lib.PROG_MSE), _envelope(model, L), f=u_data, group=group,
                         n_global=n_global)


def norm_loss(u, mode='nontrivial', eps=1e-8):
    """1/(mean u^2 + eps) or mean u^2   (Poisson_ND.py:143-147)."""
    m2 = torch.mean(u ** 2)
    if mode == 'nontrivial':
        return 1.0 / (m2 + eps)
    if mode == 'l2':
        return m2
    raise ValueError("norm mode should be 'nontrivial' or 'l2'")


def solution_jets(model, X, L, order=2):
    """(u, grad u, diag Hessian u) of ``model`` at X through the jet kernel — what
    ``model(X,L)`` + grad_scalar_field + laplacian produce (Poisson_ND.py:61-71), differentiable
    with respect to the parameters."""
    d = X.shape[1]
    J = mlp_jets(model, X, order)
    Xd = X.detach()
    N0 = J[:, 0:1]
    if getattr(model, "bc_mode", 'RB') == 'FBC':
        b = Xd * (L - Xd)
        b1 = L - 2.0 * Xd
        B = b.prod(dim=1, keepdim=True)
        excl = torch.stack([torch.cat([b[:, :i], b[:, i + 1:]], dim=1).prod(dim=1) for i in range(d)], dim=1)
        Bi, Bii = b1 * excl, -2.0 * excl
    elif getattr(model, "bc_mode", 'RB') == 'RB':
        B = torch.ones_like(N0)
        Bi = Bii = torch.zeros_like(Xd)
    else:
        raise ValueError("bc_mode must be 'FBC' or 'RB'")
    u = B * N0
    g = h = None
    if order >= 1:
        g = Bi * N0 + B * J[:, 1:1 + d]
    if order >= 2:
        h = Bii * N0 + 2.0 * Bi * J[:, 1:1 + d] + B * J[:, 1 + d:1 + 2 * d]
    return u, g, h


def grad_scalar_field(model, X, L=2.0):
    """grad u (N,d) from the jet kernel (Poisson_ND.py:61-62 takes (u, X); here the model is needed)."""
    return solution_jets(model, X, L, 1)[1]


def laplacian(model, X, L=2.0):
    """Lap u (N,1) from the jet kernel (Poisson_ND.py:64-71)."""
    return solution_jets(model, X, L, 2)[2].sum(dim=1, keepdim=True)
