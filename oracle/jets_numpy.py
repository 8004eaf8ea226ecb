"""TEST INFRASTRUCTURE ONLY — CPU oracle for the collocation-point loss step.

This module is a numpy restatement (forward-mode "jets" + hand-written reverse
sweep) of what the reference obtains with nested ``torch.autograd.grad`` calls.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline leg
may import it; the product path (the CUDA library) never does.

Parity status: PINNED.  The reference ships no golden vectors of its own
(SURVEY.md §4/§8c), so the pins are fixtures generated in the build container by
importing the reference's own functions (``tests/golden/make_golden.py`` →
``tests/golden/*.npz``); ``tests/test_oracle.py`` checks this file against them.

Reference sites restated here (paths relative to the reference checkout):
  * MLP with sin/tanh activations      Poisson_Equations/Poisson_ND.py:11-46
                                       Schrodinger_Equations/**/IPW_1D_WAN.py:62-81
  * grad / Laplacian of the network    Poisson_ND.py:61-71 (nested autograd)
  * hard-BC envelopes                  Poisson_ND.py:27-29, QHO_2D.py:149-168,
                                       IPW_1D_PINN_DRM.py:44-55, KH_1D.py:117-120
  * PINN / Deep-Ritz / Rayleigh losses Poisson_ND.py:91-103, IPW_1D_PINN_DRM.py:63-90,
                                       QHO_2D.py:363-383, KH_1D.py:226-242
  * WAN weak residual + bump weight    Poisson_ND.py:74-88,105-128, IPW_1D_WAN.py:31-59,88-115,
                                       KH_1D.py:138-148,244-269

Conventions
-----------
A network is ``Ws = [W_1 .. W_n]`` (each ``(out, in)`` like ``nn.Linear.weight``)
and ``bs = [b_1 .. b_n]``.  A *jet* of order ``o`` at a point has
``C = 1 + o*d`` channels: value, ``d`` first derivatives and (order 2) the
``d`` diagonal second derivatives.  ``J`` arrays are ``(N, C)``.
"""
from __future__ import annotations

import numpy as np

SIN, TANH = 0, 1
ENV_NONE, ENV_POLY, ENV_EXPWIN = 0, 1, 2


# --------------------------------------------------------------------------
# activation and its first three derivatives
# --------------------------------------------------------------------------
def _act(z, act):
    if act == SIN:
        s, c = np.sin(z), np.cos(z)
        return s, c, -s, -c
    if act == TANH:
        t = np.tanh(z)
        d1 = 1.0 - t * t
        d2 = -2.0 * t * d1
        d3 = -2.0 * d1 * (1.0 - 3.0 * t * t)
        return t, d1, d2, d3
    raise ValueError("activation must be SIN or TANH")


# --------------------------------------------------------------------------
# network jets: forward and reverse sweeps
# --------------------------------------------------------------------------
def mlp_jets_forward(Ws, bs, X, act=SIN, order=2):
    """Push value / gradient / Hessian-diagonal channels through the MLP.

    Returns ``(J, cache)`` with ``J`` of shape (N, 1+order*d).
    Restates Poisson_ND.py:61-71 (u, ∇u, diag ∇²u of ``model.net(X)``).
    """
    X = np.asarray(X)
    N, d = X.shape
    n = len(Ws)
    cache = {"X": X, "Z": [], "Z1": [], "Z2": [], "act": act, "order": order}
    # input jets: a = x, a'_i = e_i, a''_i = 0
    a = X
    a1 = [np.broadcast_to(np.eye(d, dtype=X.dtype)[i], (N, d)) for i in range(d)] if order >= 1 else []
    a2 = [np.zeros((N, d), dtype=X.dtype) for _ in range(d)] if order >= 2 else []
    for l in range(n):
        W, b = Ws[l], bs[l]
        z = a @ W.T + b
        z1 = [ai @ W.T for ai in a1]
        z2 = [ai @ W.T for ai in a2]
        if l == n - 1:
            J = np.concatenate([z] + z1 + z2, axis=1)
            cache["A_last"] = (a, a1, a2)
            return J, cache
        cache["Z"].append(z), cache["Z1"].append(z1), cache["Z2"].append(z2)
        if l == 0:
            cache["A_in"] = []
        cache["A_in"].append((a, a1, a2))
        s0, s1, s2, _ = _act(z, act)
        a = s0
        a1 = [s1 * zi for zi in z1]
        a2 = [s2 * z1[i] * z1[i] + s1 * z2[i] for i in range(len(z2))]
    raise AssertionError("unreachable")


def mlp_jets_backward(Ws, bs, cache, Jbar):
    """Reverse sweep: cotangents ``Jbar`` (N, C) → parameter gradients.

    Returns ``(gWs, gbs)`` = Σ_p Σ_c Jbar[p,c] ∂J[p,c]/∂θ.
    """
    X = cache["X"]
    N, d = X.shape
    act, order = cache["act"], cache["order"]
    n = len(Ws)
    gWs = [np.zeros_like(W) for W in Ws]
    gbs = [np.zeros_like(b) for b in bs]
    # split the cotangent into channels
    zb = Jbar[:, 0:1]
    zb1 = [Jbar[:, 1 + i:2 + i] for i in range(d)] if order >= 1 else []
    zb2 = [Jbar[:, 1 + d + i:2 + d + i] for i in range(d)] if order >= 2 else []
    a, a1, a2 = cache["A_last"]
    for l in range(n - 1, -1, -1):
        W = Ws[l]
        # linear layer: z_c = a_c W^T (+ b on the value channel)
        gW = zb.T @ a
        for i in range(len(zb1)):
            gW = gW + zb1[i].T @ a1[i]
        for i in range(len(zb2)):
            gW = gW + zb2[i].T @ a2[i]
        gWs[l] = gW
        gbs[l] = zb.sum(axis=0)
        if l == 0:
            break
        ab = zb @ W
        ab1 = [t @ W for t in zb1]
        ab2 = [t @ W for t in zb2]
        # activation of layer l-1
        z, z1, z2 = cache["Z"][l - 1], cache["Z1"][l - 1], cache["Z2"][l - 1]
        _, s1, s2, s3 = _act(z, act)
        zb = s1 * ab
        nzb1, nzb2 = [], []
        for i in range(len(ab1)):
            zb = zb + s2 * z1[i] * ab1[i]
            t1 = s1 * ab1[i]
            if order >= 2:
                zb = zb + (s3 * z1[i] * z1[i] + s2 * z2[i]) * ab2[i]
                t1 = t1 + 2.0 * s2 * z1[i] * ab2[i]
                nzb2.append(s1 * ab2[i])
            nzb1.append(t1)
        zb1, zb2 = nzb1, nzb2
        a, a1, a2 = cache["A_in"][l - 1]
    return gWs, gbs


# --------------------------------------------------------------------------
# separable hard-BC envelopes  B(x) = Π_i b_i(x_i)
# --------------------------------------------------------------------------
def envelope_factors(X, kind, lo=0.0, hi=2.0, nodes=None):
    """Per-dimension factor b_i(x_i) and its first two derivatives, each (N, d).

    kind ENV_POLY   : (x-lo)(hi-x)                      Poisson_ND.py:28, IPW_1D_WAN.py:79
    kind ENV_EXPWIN : (1-e^{-(x-lo)})(1-e^{x-hi})       QHO_2D.py:151-152, KH_1D.py:119 (lo=-L, hi=L)
    nodes[i]        : optional roots; factor multiplied by Π_k (x - node_k)
                      IPW_1D_PINN_DRM.py:46-51, QHO_2D.py:161-167
    """
    X = np.asarray(X)
    N, d = X.shape
    if kind == ENV_NONE:
        b = np.ones_like(X); b1 = np.zeros_like(X); b2 = np.zeros_like(X)
    elif kind == ENV_POLY:
        b = (X - lo) * (hi - X); b1 = (lo + hi) - 2.0 * X; b2 = np.full_like(X, -2.0)
    elif kind == ENV_EXPWIN:
        p = np.exp(-(X - lo)); q = np.exp(X - hi)
        b = (1.0 - p) * (1.0 - q)
        b1 = p * (1.0 - q) - (1.0 - p) * q
        b2 = -p * (1.0 - q) - 2.0 * p * q - (1.0 - p) * q
    else:
        raise ValueError("unknown envelope kind")
    if nodes is not None:
        b, b1, b2 = b.copy(), b1.copy(), b2.copy()
        for i in range(d):
            for r in (nodes[i] if i < len(nodes) else ()):
                g = X[:, i] - r
                # (b g)'' = b'' g + 2 b' ; (b g)' = b' g + b
                b2[:, i] = b2[:, i] * g + 2.0 * b1[:, i]
                b1[:, i] = b1[:, i] * g + b[:, i]
                b[:, i] = b[:, i] * g
    return b, b1, b2


def apply_envelope(J, X, order, kind, lo=0.0, hi=2.0, nodes=None):
    """u = B·N jets from network jets. Returns (U, ctx) with U shaped like J."""
    N, d = X.shape
    b, b1, b2 = envelope_factors(X, kind, lo, hi, nodes)
    B = np.prod(b, axis=1, keepdims=True)
    # exclusive products Π_{j≠i} b_j without division
    excl = np.ones_like(b)
    for i in range(d):
        for j in range(d):
            if j != i:
                excl[:, i] = excl[:, i] * b[:, j]
    Bi = b1 * excl
    Bii = b2 * excl
    U = np.empty_like(J)
    U[:, 0:1] = B * J[:, 0:1]
    if order >= 1:
        U[:, 1:1 + d] = Bi * J[:, 0:1] + B * J[:, 1:1 + d]
    if order >= 2:
        U[:, 1 + d:1 + 2 * d] = Bii * J[:, 0:1] + 2.0 * Bi * J[:, 1:1 + d] + B * J[:, 1 + d:1 + 2 * d]
    return U, (B, Bi, Bii)


def envelope_backward(Ubar, ctx, order, d):
    """Cotangent of u-jets → cotangent of network jets (envelope is parameter free)."""
    B, Bi, Bii = ctx
    Jbar = np.zeros_like(Ubar)
    Jbar[:, 0:1] = B * Ubar[:, 0:1]
    if order >= 1:
        Jbar[:, 0:1] += np.sum(Bi * Ubar[:, 1:1 + d], axis=1, keepdims=True)
        Jbar[:, 1:1 + d] = B * Ubar[:, 1:1 + d]
    if order >= 2:
        Jbar[:, 0:1] += np.sum(Bii * Ubar[:, 1 + d:1 + 2 * d], axis=1, keepdims=True)
        Jbar[:, 1:1 + d] += 2.0 * Bi * Ubar[:, 1 + d:1 + 2 * d]
        Jbar[:, 1 + d:1 + 2 * d] = B * Ubar[:, 1 + d:1 + 2 * d]
    return Jbar


# --------------------------------------------------------------------------
# residual programs on u-jets
# --------------------------------------------------------------------------
def pinn_program(U, d, f, alpha=-1.0, beta=None, E=0.0):
    """q = (alpha·Δu + (beta−E)·u − f)²  (R1).  Returns q (N,1), ∂(Σq)/∂U, ∂(Σq)/∂E.

    Poisson_ND.py:95-96 (alpha=-1), IPW_1D_PINN_DRM.py:81-82 (alpha=+1, beta=k²),
    QHO_2D.py:377-378 / KH_1D.py:233-234 (alpha=-1/2, beta=V(x), E).
    """
    u = U[:, 0:1]
    lap = np.sum(U[:, 1 + d:1 + 2 * d], axis=1, keepdims=True)
    bt = 0.0 if beta is None else beta
    r = alpha * lap + (bt - E) * u - (0.0 if f is None else f)
    q = r * r
    Ubar = np.zeros_like(U)
    Ubar[:, 0:1] = 2.0 * r * (bt - E)
    Ubar[:, 1 + d:1 + 2 * d] = 2.0 * r * alpha
    dE = float(np.sum(-2.0 * r * u))
    return q, Ubar, dE


def drm_poisson_program(U, d, f):
    """q = ½|∇u|² − f·u  (R2, Poisson_ND.py:102-103)."""
    u = U[:, 0:1]
    g = U[:, 1:1 + d]
    q = 0.5 * np.sum(g * g, axis=1, keepdims=True) - f * u
    Ubar = np.zeros_like(U)
    Ubar[:, 0:1] = -f
    Ubar[:, 1:1 + d] = g
    return q, Ubar


def rayleigh_program(U, d, a=1.0, beta=None):
    """q1 = a|∇u|² + beta·u², q2 = u²  (R3, IPW_1D_PINN_DRM.py:90, QHO_2D.py:381-383)."""
    u = U[:, 0:1]
    g = U[:, 1:1 + d]
    bt = 0.0 if beta is None else beta
    q1 = a * np.sum(g * g, axis=1, keepdims=True) + bt * u * u
    q2 = u * u
    U1 = np.zeros_like(U); U2 = np.zeros_like(U)
    U1[:, 0:1] = 2.0 * bt * u
    U1[:, 1:1 + d] = 2.0 * a * g
    U2[:, 0:1] = 2.0 * u
    return (q1, q2), (U1, U2)


def face_blocks(faces, n):
    """Axis and outward sign of each point of a blocked face batch of n points (include/pde_b200.h): face k is axis
    k // 2, sign -1 (lo) for even k and +1 (hi) for odd k; one block of n / popcount(faces) points per set bit, in
    increasing bit order.  Returns (axis, sign), each (n,)."""
    ks = [k for k in range(faces.bit_length()) if faces >> k & 1]
    per = n // len(ks)
    assert per * len(ks) == n, "n must be a multiple of popcount(faces)"
    k = np.repeat(np.array(ks), per)
    return k // 2, np.where(k % 2 == 1, 1.0, -1.0)


def flux_program(U, d, faces, f=None, alpha=1.0, beta=None):
    """q = (alpha·s·∂_a u + beta·u − f)² on a blocked face batch (PDE_PROG_FLUX, layout of face_blocks).
    Returns q (N,1) and ∂(Σq)/∂U; the program has no dq/dE."""
    u = U[:, 0:1]
    ax, s = face_blocks(faces, U.shape[0])
    rows = np.arange(U.shape[0])
    un = (s * U[rows, 1 + ax]).reshape(-1, 1)
    bt = 0.0 if beta is None else beta
    r = alpha * un + bt * u - (0.0 if f is None else f)
    Ubar = np.zeros_like(U)
    Ubar[:, 0:1] = 2.0 * r * bt
    Ubar[rows, 1 + ax] = (2.0 * r * alpha).reshape(-1) * s
    return r * r, Ubar


def ritz_value_program(U, f=None, alpha=0.0, beta=None):
    """q = ½·beta·u² − g·u with g = f, or the constant alpha when f is None (PDE_PROG_RITZ_VALUE, order 0).
    Returns q (N,1) and ∂(Σq)/∂U; the program has no dq/dE."""
    u = U[:, 0:1]
    bt = 0.0 if beta is None else beta
    g = alpha if f is None else f
    Ubar = np.zeros_like(U)
    Ubar[:, 0:1] = bt * u - g
    return 0.5 * bt * u * u - g * u, Ubar


def parabolic_program(U, d, f=None, alpha=-1.0, beta=None, E=0.0):
    """q = (∂_{d−1}u + alpha·Σ_{i<d−1} ∂²_i u + (beta−E)·u − f)², time the last coordinate (PDE_PROG_PARABOLIC, order 2).
    Returns q (N,1), ∂(Σq)/∂U and ∂(Σq)/∂E = Σ −2 r u."""
    u = U[:, 0:1]
    lap = np.sum(U[:, 1 + d:2 * d], axis=1, keepdims=True)
    bt = 0.0 if beta is None else beta
    r = U[:, d:d + 1] + alpha * lap + (bt - E) * u - (0.0 if f is None else f)
    Ubar = np.zeros_like(U)
    Ubar[:, 0:1] = 2.0 * r * (bt - E)
    Ubar[:, d:d + 1] = 2.0 * r
    Ubar[:, 1 + d:2 * d] = 2.0 * r * alpha
    return r * r, Ubar, float(np.sum(-2.0 * r * u))


def bump_weight(X, lo, hi, eps_den=0.0, I1=0.210987):
    """WAN cut-off w = Π φ(t_i), φ(t)=exp(1/(t²−1+eps_den))/I1 for |t|<1 else 0, and ∇w.

    Poisson_ND.py:74-88, IPW_1D_WAN.py:31-59 (eps_den=0); QHO_2D.py:172-202,
    KH_1D.py:138-148 (eps_den=1e-10).  At/outside the boundary both w and ∇w are 0
    (the reference's nan_to_num outcome for ∇w).
    """
    X = np.asarray(X)
    h = (hi - lo) / 2.0
    c = (hi + lo) / 2.0
    t = (X - c) / h
    inside = np.abs(t) < 1.0
    den = np.where(inside, t * t - 1.0 + eps_den, -1.0)
    phi = np.where(inside, np.exp(1.0 / den) / I1, 0.0)
    dphi = np.where(inside, phi * (-2.0 * t) / (den * den) / h, 0.0)
    w = np.prod(phi, axis=1, keepdims=True)
    d = X.shape[1]
    dw = np.empty_like(X)
    for i in range(d):
        e = np.ones(X.shape[0], dtype=X.dtype)
        for j in range(d):
            if j != i:
                e = e * phi[:, j]
        dw[:, i] = dphi[:, i] * e
    return w, dw


# --------------------------------------------------------------------------
# whole-loss helpers (value + parameter gradients), one network
# --------------------------------------------------------------------------
def _loss_and_grads(Ws, bs, X, act, order, env, program):
    J, cache = mlp_jets_forward(Ws, bs, X, act, order)
    d = X.shape[1]
    U, ctx = apply_envelope(J, X, order, env["kind"], env.get("lo", 0.0), env.get("hi", 2.0), env.get("nodes"))
    loss, Ubar, extra = program(U)
    Jbar = envelope_backward(Ubar, ctx, order, d)
    gWs, gbs = mlp_jets_backward(Ws, bs, cache, Jbar)
    return loss, gWs, gbs, extra


def poisson_pinn_loss(Ws, bs, X, f, L, bc_mode="FBC", act=SIN):
    """mean((−Δu − f)²) and its parameter gradients (Poisson_ND.py:91-96)."""
    N, d = X.shape
    env = {"kind": ENV_POLY if bc_mode == "FBC" else ENV_NONE, "lo": 0.0, "hi": L}

    def program(U):
        q, Ubar, _ = pinn_program(U, d, f, alpha=-1.0)
        return float(q.mean()), Ubar / N, None

    loss, gWs, gbs, _ = _loss_and_grads(Ws, bs, X, act, 2, env, program)
    return loss, gWs, gbs


def poisson_drm_loss(Ws, bs, X, f, L, bc_mode="FBC", act=SIN):
    """mean(½|∇u|² − f·u) and its parameter gradients (Poisson_ND.py:98-103)."""
    N, d = X.shape
    env = {"kind": ENV_POLY if bc_mode == "FBC" else ENV_NONE, "lo": 0.0, "hi": L}

    def program(U):
        q, Ubar = drm_poisson_program(U, d, f)
        return float(q.mean()), Ubar / N, None

    loss, gWs, gbs, _ = _loss_and_grads(Ws, bs, X, act, 1, env, program)
    return loss, gWs, gbs


def mse_loss(Ws, bs, X, act, env, target=None):
    """mean((u − target)²) (target None → mean(u²)) and its parameter gradients: the value-only terms of the
    reference epoch — data MSE (Poisson_ND.py:230-232), one face of boundary_loss_dirichlet (:130-141)."""
    N = X.shape[0]
    t = 0.0 if target is None else np.asarray(target, dtype=np.float64).reshape(N, 1)

    def program(U):
        r = U[:, 0:1] - t
        return float((r * r).mean()), 2.0 * r / N, None

    loss, gWs, gbs, _ = _loss_and_grads(Ws, bs, X, act, 0, env, program)
    return loss, gWs, gbs


def eigen_pinn_loss(Ws, bs, X, act, env, alpha, beta, E, f=None):
    """mean((alpha·Δu + (beta−E)u − f)²), grads and dLoss/dE (R1 general)."""
    N, d = X.shape

    def program(U):
        q, Ubar, dE = pinn_program(U, d, f, alpha=alpha, beta=beta, E=E)
        return float(q.mean()), Ubar / N, dE / N

    return _loss_and_grads(Ws, bs, X, act, 2, env, program)


def rayleigh_loss(Ws, bs, X, act, env, a, beta, eps_in=0.0, eps_out=0.0, scale=1.0):
    """(scale·m1)/(scale·(m2+eps_in)+eps_out) with m1=mean(a|∇u|²+βu²), m2=mean(u²) (R3)."""
    N, d = X.shape

    def program(U):
        (q1, q2), (U1, U2) = rayleigh_program(U, d, a, beta)
        m1, m2 = float(q1.mean()), float(q2.mean())
        den = scale * (m2 + eps_in) + eps_out
        F = scale * m1 / den
        dF1 = scale / den
        dF2 = -scale * m1 * scale / (den * den)
        return F, (dF1 * U1 + dF2 * U2) / N, (m1, m2)

    return _loss_and_grads(Ws, bs, X, act, 1, env, program)


def wan_means(u_net, v_net, X, f, lo, hi, a=1.0, beta=None, E=0.0, eps_den=0.0):
    """Per-point WAN quantities (R4) for the two networks, their means and the
    per-mean parameter-gradient vectors of both networks.

    q1 = a ∇u·∇φ + (β−E) u φ − f φ,  q2 = φ²,  q3 = u²,  q4 = |∇v|² + v²,  φ = w·v.
    Poisson_ND.py:105-128, IPW_1D_WAN.py:88-115, QHO_2D.py:204-225, KH_1D.py:244-269.
    ``u_net``/``v_net`` are dicts {Ws, bs, act, env}.  Returns
    (means[4], Gu[4] lists of (gWs, gbs), Gv[4], dq1/dE mean).
    """
    N, d = X.shape
    Ju, cu = mlp_jets_forward(u_net["Ws"], u_net["bs"], X, u_net["act"], 1)
    Jv, cv = mlp_jets_forward(v_net["Ws"], v_net["bs"], X, v_net["act"], 1)
    eu, ev = u_net["env"], v_net["env"]
    Uu, xu = apply_envelope(Ju, X, 1, eu["kind"], eu.get("lo", 0.0), eu.get("hi", 2.0), eu.get("nodes"))
    Uv, xv = apply_envelope(Jv, X, 1, ev["kind"], ev.get("lo", 0.0), ev.get("hi", 2.0), ev.get("nodes"))
    w, dw = bump_weight(X, lo, hi, eps_den)
    u, gu = Uu[:, 0:1], Uu[:, 1:]
    v, gv = Uv[:, 0:1], Uv[:, 1:]
    phi = w * v
    gphi = dw * v + w * gv
    bt = 0.0 if beta is None else beta
    ff = 0.0 if f is None else f
    q1 = a * np.sum(gu * gphi, axis=1, keepdims=True) + (bt - E) * u * phi - ff * phi
    q2 = phi * phi
    q3 = u * u
    q4 = np.sum(gv * gv, axis=1, keepdims=True) + v * v
    means = [float(q.mean()) for q in (q1, q2, q3, q4)]
    z = np.zeros_like(Uu)
    # cotangents wrt u-jets and v-jets for each q_j
    Ub = [z.copy() for _ in range(4)]
    Vb = [z.copy() for _ in range(4)]
    Ub[0][:, 0:1] = (bt - E) * phi
    Ub[0][:, 1:] = a * gphi
    Ub[2][:, 0:1] = 2.0 * u
    dq1_dphi = (bt - E) * u - ff
    dq1_dgphi = a * gu
    Vb[0][:, 0:1] = dq1_dphi * w + np.sum(dq1_dgphi * dw, axis=1, keepdims=True)
    Vb[0][:, 1:] = dq1_dgphi * w
    Vb[1][:, 0:1] = 2.0 * phi * w
    Vb[3][:, 0:1] = 2.0 * v
    Vb[3][:, 1:] = 2.0 * gv
    Gu, Gv = [], []
    for j in range(4):
        Gu.append(mlp_jets_backward(u_net["Ws"], u_net["bs"], cu, envelope_backward(Ub[j] / N, xu, 1, d)))
        Gv.append(mlp_jets_backward(v_net["Ws"], v_net["bs"], cv, envelope_backward(Vb[j] / N, xv, 1, d)))
    dE = float(np.mean(-u * phi))
    return means, Gu, Gv, dE
