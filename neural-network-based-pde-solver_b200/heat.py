"""The heat equation and other parabolic problems on the fused path (DESIGN.md §3.4c).

The reference has no time-dependent solver, so this module has no reference counterpart; it follows the conventions of
``poisson.py`` (models with ``.net`` and ``.bc_mode``, keyword-only ``group`` / ``n_global``).

Space-time points are ``X = (x_0 .. x_{d-2}, t)``: time is the LAST column, d = 2..5, and Lap_x sums over the spatial
columns only.  The interior residual is one ``PROG_PARABOLIC`` launch.  The other terms of a heat problem reuse what
exists, on the face masks below:

- initial data: ``poisson.data_loss`` (``PROG_MSE``) on points of ``initial_face(d)``;
- Dirichlet data on ``spatial_faces(d)`` points the same way, Neumann / Robin data with ``PROG_FLUX``;
- points from ``train.sample_points_rhs`` (interior) and ``train.sample_faces_rhs`` (faces).

Hard-constraint envelopes are refused: every one of them vanishes at both ends of every axis, the time axis included.
"""
from __future__ import annotations

import math

import torch

from . import _lib
from .ops import NO_ENVELOPE, ProgramSpec, residual_mean


def spatial_faces(dim):
    """Face mask of the spatial faces x_i = lo / hi, i < dim - 1, of a space-time box (include/pde_b200.h face layout:
    face k is side k % 2 of axis k // 2)."""
    return (1 << (2 * (int(dim) - 1))) - 1


def initial_face(dim):
    """Face mask of the initial face t = lo of a space-time box: bit 2 (dim - 1)."""
    return 1 << (2 * (int(dim) - 1))


def exact_u_heat(X, L, ks, kappa):
    """u*(x, t) = exp(-kappa lambda t) prod_{i < d-1} sin(k_i pi x_i / L), lambda = sum_i (k_i pi / L)^2, (N, 1).

    It solves u_t = kappa Lap_x u, vanishes on the spatial faces of [0, L]^(d-1) for integer k_i, and has the initial
    data prod_i sin(k_i pi x_i / L).  ``ks``: d - 1 wave numbers."""
    d = X.shape[1]
    if len(ks) != d - 1:
        raise ValueError(f"exact_u_heat needs {d - 1} wave numbers for {d} columns (time last), got {len(ks)}")
    lam = sum((k * math.pi / L) ** 2 for k in ks)
    u = torch.exp(-kappa * lam * X[:, d - 1:d])
    for i, k in enumerate(ks):
        u = u * torch.sin(k * math.pi * X[:, i:i + 1] / L)
    return u


def heat_residual_loss(model, X, f=None, kappa=1.0, *, group=None, n_global=None):
    """mean((u_t - kappa Lap_x u - f)^2) at the space-time points X (time last): one fused ``PROG_PARABOLIC`` launch
    (alpha = -kappa, beta = 0), differentiable w.r.t. the parameters.  ``f``: source values (N,) / (N, 1), or None for
    0.  Raises ValueError for a model with the hard-constraint envelope ('FBC') and for X with fewer than 2 columns."""
    mode = getattr(model, "bc_mode", 'RB')
    if mode == 'FBC':
        raise ValueError("heat_residual_loss: the 'FBC' envelope vanishes at t = 0 and t = L; use an 'RB' model "
                         "with initial and boundary penalties")
    if mode != 'RB':
        raise ValueError("bc_mode must be 'FBC' or 'RB'")
    if X.dim() != 2 or X.shape[1] < 2:
        raise ValueError(f"heat_residual_loss: X must be (N, d) with d >= 2 (space, then time), got {tuple(X.shape)}")
    return residual_mean(model, X, ProgramSpec(_lib.PROG_PARABOLIC, alpha=-float(kappa)), NO_ENVELOPE, f=f,
                         group=group, n_global=n_global)
