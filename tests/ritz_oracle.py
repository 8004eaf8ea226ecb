"""TEST INFRASTRUCTURE ONLY — the specification of the Ritz value program (PDE_PROG_RITZ_VALUE) and of the Deep Ritz
functional with Neumann / Robin data, in torch autograd.

The reference (Poisson_Equations/Poisson_ND.py) has only the interior half of the functional (drm_energy_loss,
:98-103), so there is no live-reference golden fixture for the boundary term: this restatement, in the style of
``oracle/autograd_ref.py`` (whose ``solution`` and ``drm_loss`` it uses), is what the kernels are tested against.
"""
from __future__ import annotations

import math

import torch

from oracle import autograd_ref as AR


def ritz_value_loss(net, X, g, L, bc_mode, kappa=0.0, alpha=0.0):
    """mean(kappa u^2 / 2 - g u) at the points X: ``g`` (N,) / (N, 1), or None for the constant ``alpha``; ``kappa`` a
    float or (N,) / (N, 1) per-point values.  No derivative of u is taken, so X need not require grad."""
    u = AR.solution(net, X, L, bc_mode)
    k = kappa.reshape(-1, 1) if torch.is_tensor(kappa) else kappa
    gv = g.reshape(-1, 1) if g is not None else alpha
    return (0.5 * k * u * u - gv * u).mean()


def boundary_energy(net, X, faces, g, L, bc_mode, kappa=0.0):
    """(popcount(faces) / L) mean(kappa u^2 / 2 - g u) on a blocked face batch: the boundary integral of the Deep Ritz
    functional over |Omega| = L^d, each of the popcount(faces) faces having area L^(d-1)."""
    return ritz_value_loss(net, X, g, L, bc_mode, kappa) * (bin(faces).count("1") / L)


def ritz_energy(net, X, f, Xb, faces, g, L, bc_mode, kappa=0.0):
    """E[u] / |Omega| on the sampled points: mean_X(|grad u|^2 / 2 - f u) + the boundary energy above."""
    return AR.drm_loss(net, X, f, L, bc_mode) + boundary_energy(net, Xb, faces, g, L, bc_mode, kappa)


def mean_value_loss(net, X, L, bc_mode, c=0.0):
    """(mean_X u - c)^2."""
    return (AR.solution(net, X, L, bc_mode).mean() - c) ** 2


def exact_mean(L, ks):
    """The mean of u* = prod_i sin(k_i pi x_i / L) over [0, L]^d: prod_i (1 - cos k_i pi) / (k_i pi)."""
    return math.prod((1.0 - math.cos(k * math.pi)) / (k * math.pi) for k in ks)
