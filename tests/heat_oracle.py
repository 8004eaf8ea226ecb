"""TEST INFRASTRUCTURE ONLY — the specification of the parabolic program (PDE_PROG_PARABOLIC) in torch autograd.

The reference has no time-dependent solver, so there is no live-reference golden fixture: this restatement, in the
style of ``oracle/autograd_ref.py`` (whose ``solution`` and first-derivative helper it uses), nests autograd once for
grad u and once more per spatial coordinate for Lap_x u.  Time is the last column of X.
"""
from __future__ import annotations

import torch

from oracle import autograd_ref as AR


def parabolic_residual(net, X, f=None, alpha=-1.0, beta=0.0, E=0.0, L=1.0, bc_mode="RB"):
    """r = du/dt + alpha Lap_x u + (beta - E) u - f at the points X (N, d), time last, (N, 1).  ``X`` must require
    grad; ``f`` (N,) / (N, 1) or None; ``beta`` a float or per-point (N,) / (N, 1); ``E`` a float or a 0-d tensor."""
    d = X.shape[1]
    u = AR.solution(net, X, L, bc_mode)
    g = AR._grad(u, X)
    lap = torch.zeros_like(u)
    for i in range(d - 1):
        lap = lap + AR._grad(g[:, i:i + 1], X)[:, i:i + 1]
    b = beta.reshape(-1, 1) if torch.is_tensor(beta) else beta
    r = g[:, d - 1:d] + alpha * lap + (b - E) * u
    if f is not None:
        r = r - f.reshape(-1, 1)
    return r


def parabolic_loss(net, X, f=None, alpha=-1.0, beta=0.0, E=0.0, L=1.0, bc_mode="RB"):
    """mean(r^2) of ``parabolic_residual``: what one PDE_PROG_PARABOLIC call returns as its mean."""
    r = parabolic_residual(net, X, f, alpha, beta, E, L, bc_mode)
    return (r * r).mean()
