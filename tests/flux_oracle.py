"""TEST INFRASTRUCTURE ONLY — the specification of the boundary-flux program (PDE_PROG_FLUX) in nested torch autograd.

The reference (Poisson_Equations/Poisson_ND.py) has no Neumann code, so there is no live-reference golden fixture for
this program: this restatement, in the style of ``oracle/autograd_ref.py`` (whose ``solution`` and ``_grad`` it uses),
is what the kernels are tested against.  Face layout as in include/pde_b200.h: face k is the side k % 2 (0: lo,
normal -e_a; 1: hi, normal +e_a) of axis a = k // 2, and a batch of N points is one equal block per set bit of the
mask, in increasing bit order.
"""
from __future__ import annotations

import math

import torch

from oracle import autograd_ref as AR


def face_list(faces):
    """The set bits of a face mask, in increasing order."""
    return [k for k in range(faces.bit_length()) if faces >> k & 1]


def normal_derivative(gu, faces):
    """n . grad u per point of a blocked face batch: gu (N, d) -> (N, 1)."""
    ks = face_list(faces)
    per = gu.shape[0] // len(ks)
    parts = [(1.0 if k % 2 else -1.0) * gu[j * per:(j + 1) * per, k // 2:k // 2 + 1] for j, k in enumerate(ks)]
    return torch.cat(parts, dim=0)


def flux_loss(net, X, faces, g, L, bc_mode, alpha=1.0, kappa=0.0):
    """mean((alpha n.grad u + kappa u - g)^2) on the blocked face batch X; ``g`` (N,) / (N, 1) or None, ``kappa`` a
    float or (N,) / (N, 1) per-point values.  X must require grad (the gradient is taken by nested autograd)."""
    u = AR.solution(net, X, L, bc_mode)
    gu = AR._grad(u, X)
    r = alpha * normal_derivative(gu, faces)
    if torch.is_tensor(kappa):
        r = r + kappa.reshape(-1, 1) * u
    elif kappa != 0.0:
        r = r + kappa * u
    if g is not None:
        r = r - g.reshape(-1, 1)
    return (r * r).mean()


def manufactured_flux(X, faces, L, ks):
    """g = s (k_a pi / L) cos(k_a pi x_a / L) prod_{j != a} sin(k_j pi x_j / L): the outward normal derivative of
    u* = prod_i sin(k_i pi x_i / L) (Poisson_ND.py:49-52) on a blocked face batch, written out (no autograd)."""
    ks_ = face_list(faces)
    per = X.shape[0] // len(ks_)
    out = []
    for j, k in enumerate(ks_):
        a, Xb = k // 2, X[j * per:(j + 1) * per]
        v = torch.ones(Xb.shape[0], dtype=X.dtype, device=X.device)
        for i, kk in enumerate(ks):
            w = kk * math.pi / L
            v = v * (w * torch.cos(w * Xb[:, i]) if i == a else torch.sin(w * Xb[:, i]))
        out.append(v if k % 2 else -v)
    return torch.cat(out)
