"""CPU tests: the oracle restatements against the golden fixtures produced by the
live reference (tests/golden/make_golden.py).  Tolerances are float64 round-off."""
import math

import numpy as np
import pytest
import torch

from conftest import assert_grads_close, flat, grads_from, load_golden, net_from, stored_entries
from oracle import autograd_ref as AR
from oracle import jets_numpy as O

TOL = 1e-11

POISSON = [
    ("poisson_pinn_d1_w64_fbc", "pinn", "FBC"), ("poisson_pinn_d3_w64_fbc", "pinn", "FBC"),
    ("poisson_drm_d5_w64_rb", "drm", "RB"), ("poisson_pinn_d2_w16_fbc", "pinn", "FBC"),
    ("poisson_pinn_d5_w16_fbc", "pinn", "FBC"), ("poisson_pinn_d3_w16_rb", "pinn", "RB"),
    ("poisson_pinn_d4_w12_fbc", "pinn", "FBC"), ("poisson_drm_d1_w16_fbc", "drm", "FBC"),
    ("poisson_drm_d2_w16_fbc", "drm", "FBC"), ("poisson_drm_d3_w16_fbc", "drm", "FBC"),
]


@pytest.mark.parametrize("name,method,bc", POISSON)
def test_numpy_oracle_poisson(name, method, bc):
    g = load_golden(name)
    Ws, bs = net_from(g)
    fn = O.poisson_pinn_loss if method == "pinn" else O.poisson_drm_loss
    loss, gWs, gbs = fn(Ws, bs, g["X"], g["f"], float(g["L"]), bc)
    assert abs(loss - g["loss"]) <= TOL * max(1.0, abs(g["loss"]))
    assert_grads_close((gWs, gbs), grads_from(g), TOL, name)


@pytest.mark.parametrize("name,method,bc", POISSON)
def test_numpy_oracle_jets(name, method, bc):
    """u, grad u and Laplacian from the jets equal the reference helpers' outputs."""
    g = load_golden(name)
    Ws, bs = net_from(g)
    X = g["X"]; d = X.shape[1]
    J, _ = O.mlp_jets_forward(Ws, bs, X, O.SIN, 2)
    U, _ = O.apply_envelope(J, X, 2, O.ENV_POLY if bc == "FBC" else O.ENV_NONE, 0.0, float(g["L"]))
    np.testing.assert_allclose(U[:, 0:1], g["u"], rtol=0, atol=TOL * max(1, np.abs(g["u"]).max()))
    np.testing.assert_allclose(U[:, 1:1 + d], g["grad_u"], rtol=0, atol=TOL * max(1, np.abs(g["grad_u"]).max()))
    np.testing.assert_allclose(U[:, 1 + d:].sum(1, keepdims=True), g["lap_u"], rtol=0, atol=TOL * max(1, np.abs(g["lap_u"]).max()))


@pytest.mark.parametrize("name,method,bc", POISSON[:6])
def test_autograd_port_poisson(name, method, bc):
    g = load_golden(name)
    Ws, bs = net_from(g)
    widths = [Ws[0].shape[1]] + [W.shape[0] for W in Ws]
    net = AR.build_mlp(widths, "sin", torch.float64)
    AR.load_params(net, Ws, bs)
    X = torch.tensor(g["X"]); f = torch.tensor(g["f"])
    loss, gflat = AR.loss_and_grads(method, net, X, f, float(g["L"]), bc)
    assert abs(loss - g["loss"]) <= TOL * max(1.0, abs(g["loss"]))
    want = flat(*grads_from(g))
    assert np.max(np.abs(gflat.numpy() - want)) <= TOL * np.max(np.abs(want))
    # chunked accumulation (how the CPU baseline handles 2^22 points) is exact for plain means
    loss2, g2 = AR.loss_and_grads(method, net, X, f, float(g["L"]), bc, chunk=17)
    assert abs(loss2 - g["loss"]) <= 1e-11 * max(1.0, abs(g["loss"]))
    assert np.max(np.abs(g2.numpy() - want)) <= 1e-11 * np.max(np.abs(want))


def test_network_free_known_answer():
    """-Δu* == f for the manufactured solution (Poisson_ND.py:49-58): pins the rhs helper."""
    torch.manual_seed(3)
    L, ks = 2.0, [1, 2, 3]
    X = (torch.rand(200, 3, dtype=torch.float64) * L).requires_grad_(True)
    u = torch.ones(200, 1, dtype=torch.float64)
    for i, k in enumerate(ks):
        u = u * torch.sin(k * math.pi * X[:, i:i + 1] / L)
    lap = AR._laplace(u, X)
    assert (-lap - AR.manufactured_rhs(X, L, ks)).abs().max().item() < 5e-12


def _wan_check(g, u_net, v_net, X, f, lo, hi, a, beta, E, eps_den):
    return O.wan_means(u_net, v_net, X, f, lo, hi, a=a, beta=beta, E=E, eps_den=eps_den)


def _combine(G, coefs):
    gW = [sum(c * G[j][0][i] for j, c in enumerate(coefs)) for i in range(len(G[0][0]))]
    gb = [sum(c * G[j][1][i] for j, c in enumerate(coefs)) for i in range(len(G[0][1]))]
    return gW, gb


def test_numpy_oracle_poisson_wan():
    g = load_golden("poisson_wan_d2_w16")
    L = float(g["L"]); eps = 1e-8; reg = float(g["v_reg_weight"])
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    u_net = dict(Ws=uW, bs=ub, act=O.SIN, env=dict(kind=O.ENV_POLY, lo=0.0, hi=L))
    v_net = dict(Ws=vW, bs=vb, act=O.SIN, env=dict(kind=O.ENV_NONE))
    m, Gu, Gv, _ = O.wan_means(u_net, v_net, g["X"], g["f"], 0.0, L, a=1.0)
    m1, m2, m3, m4 = m
    loss_u = m1 * m1 / (m2 + eps)
    loss_v = -math.log(loss_u + eps) + reg * m4
    assert abs(m1 - g["weak"]) <= TOL and abs(m2 - g["phi_norm"]) <= TOL
    assert abs(loss_u - g["loss_u"]) <= TOL * max(1, abs(g["loss_u"]))
    assert abs(loss_v - g["loss_v"]) <= TOL * max(1, abs(g["loss_v"]))
    dlu = [2 * m1 / (m2 + eps), -m1 * m1 / (m2 + eps) ** 2, 0.0, 0.0]
    k = -1.0 / (loss_u + eps)
    dlv = [k * dlu[0], k * dlu[1], 0.0, reg]
    assert_grads_close(_combine(Gu, dlu), grads_from(g, "lu_u_"), 1e-11, "lu/u")
    assert_grads_close(_combine(Gv, dlu), grads_from(g, "lu_v_"), 1e-11, "lu/v")
    assert_grads_close(_combine(Gu, dlv), grads_from(g, "lv_u_"), 1e-11, "lv/u")
    assert_grads_close(_combine(Gv, dlv), grads_from(g, "lv_v_"), 1e-11, "lv/v")


@pytest.mark.parametrize("name", ["ipw1d_fbc_n2", "ipw1d_fn_n3"])
def test_numpy_oracle_ipw1d(name):
    g = load_golden(name)
    Ws, bs = net_from(g)
    L = float(g["L"]); n = int(g["n"]); X = g["x"]
    # the reference stores node positions as float32 tensors (IPW_1D_PINN_DRM.py:38-40)
    nodes = [[float(np.float32(k * L / n)) for k in range(1, n)]] if name.endswith("fn_n3") else None
    env = dict(kind=O.ENV_POLY, lo=0.0, hi=L, nodes=nodes)
    k2 = (n * math.pi / L) ** 2
    loss, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, O.TANH, env, alpha=1.0, beta=k2, E=0.0)
    assert abs(loss - g["pinn_loss"]) <= 1e-11 * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), 1e-11, name + " pinn")
    loss, gWs, gbs, _ = O.rayleigh_loss(Ws, bs, X, O.TANH, env, a=1.0, beta=None)
    assert abs(loss - g["drm_loss"]) <= 1e-11 * max(1, abs(g["drm_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "drm_"), 1e-11, name + " drm")


def test_numpy_oracle_ipw1d_wan():
    g = load_golden("ipw1d_wan_n2")
    L = float(g["L"]); n = int(g["n"]); X = g["x"]
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    u_net = dict(Ws=uW, bs=ub, act=O.TANH, env=dict(kind=O.ENV_POLY, lo=0.0, hi=L))
    v_net = dict(Ws=vW, bs=vb, act=O.TANH, env=dict(kind=O.ENV_NONE))
    E = (n * math.pi) ** 2 / (2 * L * L)
    m, Gu, Gv, _ = O.wan_means(u_net, v_net, X, None, 0.0, L, a=0.5, beta=None, E=E)
    m1, m2, m3, _ = m
    lpde = m1 * m1 / (m2 + 1e-8)
    lnorm = (L * m3 - 1.0) ** 2
    assert abs(lpde - g["loss_pde"]) <= 1e-11 * max(1, abs(g["loss_pde"]))
    assert abs(lnorm - g["loss_norm"]) <= 1e-11 * max(1, abs(g["loss_norm"]))
    dtot = [2 * m1 / (m2 + 1e-8), -m1 * m1 / (m2 + 1e-8) ** 2, 2 * (L * m3 - 1.0) * L, 0.0]
    k = -1.0 / (lpde + 1e-8)
    dlv = [k * dtot[0], k * dtot[1], 0.0, 0.0]
    assert_grads_close(_combine(Gu, dtot), grads_from(g, "tot_u_"), 1e-11, "tot/u")
    assert_grads_close(_combine(Gv, dtot), grads_from(g, "tot_v_"), 1e-11, "tot/v")
    assert_grads_close(_combine(Gu, dlv), grads_from(g, "lv_u_"), 1e-11, "lv/u")
    assert_grads_close(_combine(Gv, dlv), grads_from(g, "lv_v_"), 1e-11, "lv/v")


@pytest.mark.parametrize("name", ["qho2d_fbc_00", "qho2d_fn_21"])
def test_numpy_oracle_qho2d(name):
    g = load_golden(name)
    Ws, bs = net_from(g)
    L = float(g["L"]); E = float(g["E"])
    X = np.stack([g["x"].reshape(-1), g["y"].reshape(-1)], axis=1)
    nodes = [list(g["nodes_x"]), list(g["nodes_y"])] if "fn" in name else None
    env = dict(kind=O.ENV_EXPWIN, lo=-L, hi=L, nodes=nodes)
    V = 0.5 * math.sqrt(2) ** 2 * (X[:, 0:1] ** 2 + X[:, 1:2] ** 2)
    J, _ = O.mlp_jets_forward(Ws, bs, X, O.SIN, 0)
    U, _ = O.apply_envelope(J, X, 0, env["kind"], -L, L, nodes)
    np.testing.assert_allclose(U.reshape(g["u"].shape), g["u"], rtol=0, atol=1e-11 * max(1, np.abs(g["u"]).max()))
    loss, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, O.SIN, env, alpha=-0.5, beta=V, E=E)
    assert abs(loss - g["pinn_loss"]) <= 1e-11 * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), 1e-11, name + " pinn")
    loss, gWs, gbs, _ = O.rayleigh_loss(Ws, bs, X, O.SIN, env, a=0.5, beta=V, eps_in=1e-8)
    assert abs(loss - g["drm_loss"]) <= 1e-11 * max(1, abs(g["drm_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "drm_"), 1e-11, name + " drm")


def test_numpy_oracle_qho2d_wan():
    g = load_golden("qho2d_wan_10")
    L = float(g["L"]); E = float(g["E"])
    X = np.stack([g["x"].reshape(-1), g["y"].reshape(-1)], axis=1)
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    env = dict(kind=O.ENV_EXPWIN, lo=-L, hi=L)
    u_net = dict(Ws=uW, bs=ub, act=O.SIN, env=env)
    v_net = dict(Ws=vW, bs=vb, act=O.SIN, env=env)
    V = 0.5 * math.sqrt(2) ** 2 * (X[:, 0:1] ** 2 + X[:, 1:2] ** 2)
    m, Gu, Gv, _ = O.wan_means(u_net, v_net, X, None, -L, L, a=0.5, beta=V, E=E, eps_den=1e-10)
    m1, m2, m3, _ = m
    lpde = m1 * m1 / (m2 + 1e-8)
    lnorm = (4 * L * L * m3 - 1.0) ** 2
    assert abs(lpde - g["loss_pde"]) <= 1e-11 * max(1, abs(g["loss_pde"]))
    assert abs(lnorm - g["loss_norm"]) <= 1e-11 * max(1, abs(g["loss_norm"]))
    dtot = [2 * m1 / (m2 + 1e-8), -m1 * m1 / (m2 + 1e-8) ** 2, 2 * (4 * L * L * m3 - 1.0) * 4 * L * L, 0.0]
    assert_grads_close(_combine(Gu, dtot), grads_from(g, "tot_u_"), 1e-11, "tot/u")
    assert_grads_close(_combine(Gv, dtot), grads_from(g, "tot_v_"), 1e-11, "tot/v")


@pytest.mark.parametrize("name,kind", [("kh1d_raw", O.ENV_NONE), ("kh1d_fbc", O.ENV_EXPWIN)])
def test_numpy_oracle_kh1d(name, kind):
    g = load_golden(name)
    L = float(g["L"]); E = float(g["E"])
    X = g["x"].reshape(-1, 1); V = g["V"].reshape(-1, 1)
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    # pinn_loss uses L_here = max|x| (KH_1D.py:227) which equals L on this grid
    env = dict(kind=kind, lo=-L, hi=L)
    loss, gWs, gbs, dE = O.eigen_pinn_loss(uW, ub, X, O.SIN, env, alpha=-0.5, beta=V, E=E)
    assert abs(loss - g["pinn_loss"]) <= 1e-11 * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), 1e-11, name + " pinn")
    assert abs(dE - float(g["pinn_gE"])) <= 1e-11 * max(1, abs(float(g["pinn_gE"])))
    loss, gWs, gbs, _ = O.rayleigh_loss(uW, ub, X, O.SIN, env, a=0.5, beta=V, eps_out=1e-12, scale=2 * L)
    assert abs(loss - g["drm_loss"]) <= 1e-11 * max(1, abs(g["drm_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "drm_"), 1e-11, name + " drm")
    # wan: pde = (2L m1 / (2L m2 + 1e-12))², norm = (2L m3 − 1)²; v-net is RAW FCN1D
    u_net = dict(Ws=uW, bs=ub, act=O.SIN, env=env)
    v_net = dict(Ws=vW, bs=vb, act=O.SIN, env=dict(kind=O.ENV_NONE))
    m, Gu, Gv, dE1 = O.wan_means(u_net, v_net, X, None, -L, L, a=0.5, beta=V, E=E, eps_den=1e-10)
    m1, m2, m3, _ = m
    den = 2 * L * m2 + 1e-12
    ratio = 2 * L * m1 / den
    pde = ratio ** 2
    nrm = (2 * L * m3 - 1.0) ** 2
    assert abs(pde - g["wan_pde"]) <= 1e-11 * max(1, abs(g["wan_pde"]))
    assert abs(nrm - g["wan_norm"]) <= 1e-11 * max(1, abs(g["wan_norm"]))
    d = [2 * ratio * 2 * L / den, -2 * ratio * 2 * L * m1 * 2 * L / den ** 2, 2 * (2 * L * m3 - 1.0) * 2 * L, 0.0]
    assert_grads_close(_combine(Gu, d), grads_from(g, "wan_u_"), 1e-11, "wan/u")
    assert_grads_close(_combine(Gv, d), grads_from(g, "wan_v_"), 1e-11, "wan/v")
    assert abs(d[0] * dE1 - float(g["wan_gE"])) <= 1e-11 * max(1, abs(float(g["wan_gE"])))


# ---------------------------------------------------------------- second fixture set (make_golden.py more)
def _qho1d_env(name, X_max, n):
    from_nodes = {2: [-2 ** (-3 / 4), 2 ** (-3 / 4)], 3: [0.0, -2 ** (-3 / 4) * math.sqrt(3), 2 ** (-3 / 4) * math.sqrt(3)]}
    nodes = [[float(np.float32(v)) for v in from_nodes[n]]] if "fn" in name else None   # float32 tensors in the reference
    kind = O.ENV_NONE if "fnonly" in name else O.ENV_EXPWIN
    return dict(kind=kind, lo=-X_max, hi=X_max, nodes=nodes)


@pytest.mark.parametrize("name", ["qho1d_bc_n1", "qho1d_fn_n2", "qho1d_fnonly_n3"])
def test_numpy_oracle_qho1d(name):
    """QHO_1D_PINN_DRM.py:161-185 (ModuleList sine network, exp window and / or forced nodes)."""
    g = load_golden(name)
    Ws, bs = net_from(g)
    X_max, n, X = float(g["X_max"]), int(g["n"]), g["x"]
    env = _qho1d_env(name, X_max, n)
    V = X ** 2          # 1/2 omega^2 x^2, omega = sqrt 2
    loss, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, O.SIN, env, alpha=-0.5, beta=V, E=(n + 0.5) * math.sqrt(2))
    assert abs(loss - g["pinn_loss"]) <= 1e-11 * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), 1e-11, name + " pinn")
    loss, gWs, gbs, _ = O.rayleigh_loss(Ws, bs, X, O.SIN, env, a=0.5, beta=V)
    assert abs(loss - g["drm_loss"]) <= 1e-11 * max(1, abs(g["drm_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "drm_"), 1e-11, name + " drm")
    # value-only terms: (sqrt(sum u^2 dx) - 1)^2
    J, _ = O.mlp_jets_forward(Ws, bs, X, O.SIN, 0)
    U, _ = O.apply_envelope(J, X, 0, env["kind"], -X_max, X_max, env["nodes"])
    dx = X[1, 0] - X[0, 0]
    assert abs((math.sqrt((U ** 2).sum() * dx) - 1) ** 2 - g["norm_loss"]) <= 1e-11 * max(1, abs(g["norm_loss"]))


def test_numpy_oracle_qho1d_wan():
    """QHO_1D_WAN.py:115-140 with the trainable energy."""
    g = load_golden("qho1d_wan_n1")
    L, E, X = float(g["L"]), float(g["E"]), g["x"]
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    u_net = dict(Ws=uW, bs=ub, act=O.TANH, env=dict(kind=O.ENV_EXPWIN, lo=-L, hi=L))
    v_net = dict(Ws=vW, bs=vb, act=O.TANH, env=dict(kind=O.ENV_NONE))
    m, Gu, Gv, dE1 = O.wan_means(u_net, v_net, X, None, -L, L, a=0.5, beta=X ** 2, E=E)
    m1, m2, m3, _ = m
    lpde = m1 * m1 / (m2 + 1e-8)
    lnorm = (2 * L * m3 - 1.0) ** 2
    assert abs(lpde - g["loss_pde"]) <= 1e-11 * max(1, abs(g["loss_pde"]))
    assert abs(lnorm - g["loss_norm"]) <= 1e-11 * max(1, abs(g["loss_norm"]))
    dtot = [2 * m1 / (m2 + 1e-8), -m1 * m1 / (m2 + 1e-8) ** 2, 2 * (2 * L * m3 - 1.0) * 2 * L, 0.0]
    assert_grads_close(_combine(Gu, dtot), grads_from(g, "tot_u_"), 1e-11, "tot/u")
    assert_grads_close(_combine(Gv, dtot), grads_from(g, "tot_v_"), 1e-11, "tot/v")
    assert abs(dtot[0] * dE1 - float(g["tot_gE"])) <= 1e-8 * max(1, abs(float(g["tot_gE"])))


def test_numpy_oracle_ipw1d_wan_fn():
    """IPW_1D_WAN_FN.py:91-118: forced nodes j L / n on u (n = 3) and none on v (n = 1)."""
    g = load_golden("ipw1d_wanfn_n3")
    L, n, X = float(g["L"]), int(g["n"]), g["x"]
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    u_net = dict(Ws=uW, bs=ub, act=O.TANH, env=dict(kind=O.ENV_POLY, lo=0.0, hi=L, nodes=[[j * L / n for j in range(1, n)]]))
    v_net = dict(Ws=vW, bs=vb, act=O.TANH, env=dict(kind=O.ENV_POLY, lo=0.0, hi=L))
    E = (n * math.pi) ** 2 / (2 * L * L)
    m, Gu, Gv, _ = O.wan_means(u_net, v_net, X, None, 0.0, L, a=0.5, beta=None, E=E)
    m1, m2, m3, _ = m
    lpde = m1 * m1 / (m2 + 1e-8)
    lnorm = (L * m3 - 1.0) ** 2
    assert abs(lpde - g["loss_pde"]) <= 1e-11 * max(1, abs(g["loss_pde"]))
    assert abs(lnorm - g["loss_norm"]) <= 1e-11 * max(1, abs(g["loss_norm"]))
    dtot = [2 * m1 / (m2 + 1e-8), -m1 * m1 / (m2 + 1e-8) ** 2, 2 * (L * m3 - 1.0) * L, 0.0]
    assert_grads_close(_combine(Gu, dtot), grads_from(g, "tot_u_"), 1e-11, "tot/u")
    assert_grads_close(_combine(Gv, dtot), grads_from(g, "tot_v_"), 1e-11, "tot/v")


@pytest.mark.parametrize("name", ["ipw2d_fbc_11", "ipw2d_fn_32"])
def test_numpy_oracle_ipw2d(name):
    """IPW_2D.py:195-228 inline PINN / DRM blocks."""
    g = load_golden(name)
    Ws, bs = net_from(g)
    L, nx, ny = float(g["L"]), int(g["nx"]), int(g["ny"])
    X = np.stack([g["x"].reshape(-1), g["y"].reshape(-1)], axis=1)
    nodes = [[k * L / nx for k in range(1, nx)], [k * L / ny for k in range(1, ny)]] if "fn" in name else None
    env = dict(kind=O.ENV_POLY, lo=0.0, hi=L, nodes=nodes)
    k2 = (nx * math.pi / L) ** 2 + (ny * math.pi / L) ** 2
    loss, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, O.SIN, env, alpha=1.0, beta=k2, E=0.0)
    assert abs(loss - g["pinn_loss"]) <= 1e-11 * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), 1e-11, name + " pinn")
    loss, gWs, gbs, _ = O.rayleigh_loss(Ws, bs, X, O.SIN, env, a=1.0, beta=None, eps_in=1e-8)
    assert abs(loss - g["drm_loss"]) <= 1e-11 * max(1, abs(g["drm_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "drm_"), 1e-11, name + " drm")


def test_numpy_oracle_qho2d_energy():
    """QHO_2D_Energy.py:382-383: dLoss/dE of the PINN residual with a trainable energy."""
    g = load_golden("qho2d_energy_11")
    Ws, bs = net_from(g)
    L, E = float(g["L"]), float(g["E"])
    X = np.stack([g["x"].reshape(-1), g["y"].reshape(-1)], axis=1)
    V = X[:, 0:1] ** 2 + X[:, 1:2] ** 2
    loss, gWs, gbs, dE = O.eigen_pinn_loss(Ws, bs, X, O.SIN, dict(kind=O.ENV_EXPWIN, lo=-L, hi=L), alpha=-0.5, beta=V, E=E)
    assert abs(loss - g["pinn_loss"]) <= 1e-11 * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), 1e-11, "qho2d energy pinn")
    assert abs(dE - float(g["pinn_gE"])) <= 1e-11 * max(1, abs(float(g["pinn_gE"])))


# ---------------------------------------------------------------- value-only terms and the config-shaped fixtures
def test_numpy_oracle_value_terms():
    """Data MSE, both norm_loss modes and the Dirichlet face penalty (Poisson_ND.py:130-147,230-239)."""
    g = load_golden("poisson_value_terms_d3_w16_rb")
    Ws, bs = net_from(g)
    env = dict(kind=O.ENV_NONE)
    loss, gWs, gbs = O.mse_loss(Ws, bs, g["Xd"], O.SIN, env, g["ud"])
    assert abs(loss - g["data_loss"]) <= TOL * max(1, abs(g["data_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "data_"), TOL, "data")
    m2, gW2, gb2 = O.mse_loss(Ws, bs, g["Xd"], O.SIN, env, None)
    for mode, F, dF in (("nontrivial", 1.0 / (m2 + 1e-8), -1.0 / (m2 + 1e-8) ** 2), ("l2", m2, 1.0)):
        assert abs(F - g[f"norm_{mode}_loss"]) <= TOL * max(1, abs(g[f"norm_{mode}_loss"]))
        assert_grads_close(([dF * a for a in gW2], [dF * a for a in gb2]), grads_from(g, f"norm_{mode}_"), TOL, mode)
    nf = g["Xb"].shape[0]
    tot, gW, gb = 0.0, [np.zeros_like(W) for W in Ws], [np.zeros_like(b) for b in bs]
    for Xb in g["Xb"]:
        l, a, b = O.mse_loss(Ws, bs, Xb, O.SIN, env, None)
        tot += l / nf
        gW = [x + y / nf for x, y in zip(gW, a)]; gb = [x + y / nf for x, y in zip(gb, b)]
    assert abs(tot - g["bc_loss"]) <= TOL * max(1, abs(g["bc_loss"]))
    assert_grads_close((gW, gb), grads_from(g, "bc_"), TOL, "bc")


def _grid_points(g, lo):
    L = float(g["L"])
    g1 = np.linspace(lo, L, int(g["grid_n"]))
    xg, yg = np.meshgrid(g1, g1, indexing="ij")
    return np.stack([xg.reshape(-1), yg.reshape(-1)], axis=1)


@pytest.mark.parametrize("name", ["cfg4_qho2d_fbc_00", "cfg4_qho2d_fn_21"])
def test_numpy_oracle_config4_qho2d(name):
    """BASELINE config 4 at its own shape: QHO_2D.FCN([2,50,50,50,50,1]) on the 200 x 200 grid (QHO_2D.py:249-254,281)."""
    g = load_golden(name)
    Ws, bs = net_from(g)
    L, E = float(g["L"]), float(g["E"])
    X = _grid_points(g, -L)
    assert X.shape[0] == 40000 and [W.shape[0] for W in Ws] == [50, 50, 50, 50, 1]
    nodes = [list(g["nodes_x"]), list(g["nodes_y"])] if "fn" in name else None
    env = dict(kind=O.ENV_EXPWIN, lo=-L, hi=L, nodes=nodes)
    V = 0.5 * math.sqrt(2) ** 2 * (X[:, 0:1] ** 2 + X[:, 1:2] ** 2)
    loss, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, O.SIN, env, alpha=-0.5, beta=V, E=E)
    assert abs(loss - g["pinn_loss"]) <= TOL * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), TOL, name + " pinn")
    loss, gWs, gbs, _ = O.rayleigh_loss(Ws, bs, X, O.SIN, env, a=0.5, beta=V, eps_in=1e-8)
    assert abs(loss - g["drm_loss"]) <= TOL * max(1, abs(g["drm_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "drm_"), TOL, name + " drm")


@pytest.mark.parametrize("name", ["cfg4_ipw2d_fbc_11", "cfg4_ipw2d_fn_32"])
def test_numpy_oracle_config4_ipw2d(name):
    """IPW_2D.FCN([2,50,50,50,50,1]) on the 200 x 200 grid (IPW_2D.py:137-138,166,195-228)."""
    g = load_golden(name)
    Ws, bs = net_from(g)
    L, nx, ny = float(g["L"]), int(g["nx"]), int(g["ny"])
    X = _grid_points(g, 0.0)
    nodes = None
    if "fn" in name:   # Python-float node positions k L / n (IPW_2D.py:101-107)
        nodes = [[k * L / n for k in range(1, n)] for n in (nx, ny)]
    env = dict(kind=O.ENV_POLY, lo=0.0, hi=L, nodes=nodes)
    k2 = 2 * ((nx * np.pi) ** 2 / (2 * L ** 2) + (ny * np.pi) ** 2 / (2 * L ** 2))
    loss, gWs, gbs, _ = O.eigen_pinn_loss(Ws, bs, X, O.SIN, env, alpha=1.0, beta=k2, E=0.0)
    assert abs(loss - g["pinn_loss"]) <= TOL * max(1, abs(g["pinn_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "pinn_"), TOL, name + " pinn")
    loss, gWs, gbs, _ = O.rayleigh_loss(Ws, bs, X, O.SIN, env, a=1.0, beta=None, eps_in=1e-8)
    assert abs(loss - g["drm_loss"]) <= TOL * max(1, abs(g["drm_loss"]))
    assert_grads_close((gWs, gbs), grads_from(g, "drm_"), TOL, name + " drm")


def _wan_dtot(m1, m2, m3, vol):
    return [2 * m1 / (m2 + 1e-8), -m1 * m1 / (m2 + 1e-8) ** 2, 2 * (vol * m3 - 1.0) * vol, 0.0]


def test_numpy_oracle_config4_qho2d_wan():
    g = load_golden("cfg4_qho2d_wan_10")
    L, E = float(g["L"]), float(g["E"])
    X = _grid_points(g, -L)
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    env = dict(kind=O.ENV_EXPWIN, lo=-L, hi=L)
    V = 0.5 * math.sqrt(2) ** 2 * (X[:, 0:1] ** 2 + X[:, 1:2] ** 2)
    m, Gu, Gv, _ = O.wan_means(dict(Ws=uW, bs=ub, act=O.SIN, env=env), dict(Ws=vW, bs=vb, act=O.SIN, env=env), X, None,
                               -L, L, a=0.5, beta=V, E=E, eps_den=1e-10)
    m1, m2, m3, _ = m
    assert abs(m1 * m1 / (m2 + 1e-8) - g["loss_pde"]) <= TOL * max(1, abs(g["loss_pde"]))
    assert abs((4 * L * L * m3 - 1.0) ** 2 - g["loss_norm"]) <= TOL * max(1, abs(g["loss_norm"]))
    dtot = _wan_dtot(m1, m2, m3, 4 * L * L)
    assert_grads_close(_combine(Gu, dtot), grads_from(g, "tot_u_"), TOL, "tot/u")
    assert_grads_close(_combine(Gv, dtot), grads_from(g, "tot_v_"), TOL, "tot/v")


def test_numpy_oracle_config5_ipw1d_wan():
    """IPW_1D_WAN at its own shape: u [1,50,50,50,1] / v [1,20,20,20,1], linspace(0, 2, 1000) (IPW_1D_WAN.py:140-166)."""
    g = load_golden("cfg5_ipw1d_wan_n2")
    L, n, X = float(g["L"]), int(g["n"]), g["x"]
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    assert X.shape[0] == 1000 and [W.shape[0] for W in uW] == [50, 50, 50, 1] and [W.shape[0] for W in vW] == [20, 20, 20, 1]
    u_net = dict(Ws=uW, bs=ub, act=O.TANH, env=dict(kind=O.ENV_POLY, lo=0.0, hi=L))
    v_net = dict(Ws=vW, bs=vb, act=O.TANH, env=dict(kind=O.ENV_NONE))
    m, Gu, Gv, _ = O.wan_means(u_net, v_net, X, None, 0.0, L, a=0.5, beta=None, E=(n * math.pi) ** 2 / (2 * L * L))
    m1, m2, m3, _ = m
    lpde = m1 * m1 / (m2 + 1e-8)
    assert abs(lpde - g["loss_pde"]) <= TOL * max(1, abs(g["loss_pde"]))
    assert abs((L * m3 - 1.0) ** 2 - g["loss_norm"]) <= TOL * max(1, abs(g["loss_norm"]))
    dtot = _wan_dtot(m1, m2, m3, L)
    k = -1.0 / (lpde + 1e-8)
    assert_grads_close(_combine(Gu, dtot), grads_from(g, "tot_u_"), TOL, "tot/u")
    assert_grads_close(_combine(Gv, dtot), grads_from(g, "tot_v_"), TOL, "tot/v")
    assert_grads_close(_combine(Gv, [k * dtot[0], k * dtot[1], 0.0, 0.0]), grads_from(g, "lv_v_"), TOL, "lv/v")


def test_numpy_oracle_config5_kh1d():
    """KH_1D at its own shape (KH_1D.py:624-638): u [1,100,100,100,1], v [1,50,50,50,1], 1024 points on [-60, 60], alpha = 10."""
    g = load_golden("cfg5_kh1d_a10")
    L, E = float(g["L"]), float(g["E"])
    X = g["x"].reshape(-1, 1); V = g["V"].reshape(-1, 1)
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_"); wW, wb = net_from(g, "w_")
    assert X.shape[0] == 1024 and [W.shape[0] for W in uW] == [100, 100, 100, 1]
    env = dict(kind=O.ENV_EXPWIN, lo=-L, hi=L)
    loss, gWs, gbs, dE = O.eigen_pinn_loss(uW, ub, X, O.SIN, env, alpha=-0.5, beta=V, E=E)
    assert abs(loss - g["pinn_loss"]) <= TOL * max(1, abs(g["pinn_loss"]))
    assert_grads_close(stored_entries((gWs, gbs), g, "pinn_"), grads_from(g, "pinn_"), TOL, "pinn")
    assert abs(dE - float(g["pinn_gE"])) <= TOL * max(1, abs(float(g["pinn_gE"])))
    loss, gWs, gbs, _ = O.rayleigh_loss(uW, ub, X, O.SIN, env, a=0.5, beta=V, eps_out=1e-12, scale=2 * L)
    assert abs(loss - g["drm_loss"]) <= TOL * max(1, abs(g["drm_loss"]))
    assert_grads_close(stored_entries((gWs, gbs), g, "drm_"), grads_from(g, "drm_"), TOL, "drm")
    raw = dict(kind=O.ENV_NONE)
    m, Gu, Gv, dE1 = O.wan_means(dict(Ws=wW, bs=wb, act=O.SIN, env=raw), dict(Ws=vW, bs=vb, act=O.SIN, env=raw), X, None,
                                 -L, L, a=0.5, beta=V, E=E, eps_den=1e-10)
    m1, m2, m3, _ = m
    den = 2 * L * m2 + 1e-12
    ratio = 2 * L * m1 / den
    assert abs(ratio ** 2 - g["wan_pde"]) <= TOL * max(1, abs(g["wan_pde"]))
    assert abs((2 * L * m3 - 1.0) ** 2 - g["wan_norm"]) <= TOL * max(1, abs(g["wan_norm"]))
    d = [2 * ratio * 2 * L / den, -2 * ratio * 2 * L * m1 * 2 * L / den ** 2, 2 * (2 * L * m3 - 1.0) * 2 * L, 0.0]
    assert_grads_close(stored_entries(_combine(Gu, d), g, "wan_u_"), grads_from(g, "wan_u_"), TOL, "wan/u")
    assert_grads_close(stored_entries(_combine(Gv, d), g, "wan_v_"), grads_from(g, "wan_v_"), TOL, "wan/v")
    assert abs(d[0] * dE1 - float(g["wan_gE"])) <= TOL * max(1, abs(float(g["wan_gE"])))


def test_numpy_oracle_config5_qho1d_wan():
    """QHO_1D_WAN at its own shape (QHO_1D_WAN.py:159,169-176): u [1,200,200,200,1], v [1,100,100,100,1], 1000 points."""
    g = load_golden("cfg5_qho1d_wan_n1")
    L, E, X = float(g["L"]), float(g["E"]), g["x"]
    uW, ub = net_from(g, "u_"); vW, vb = net_from(g, "v_")
    assert [W.shape[0] for W in uW] == [200, 200, 200, 1] and [W.shape[0] for W in vW] == [100, 100, 100, 1]
    env = dict(kind=O.ENV_EXPWIN, lo=-L, hi=L)
    m, Gu, Gv, dE1 = O.wan_means(dict(Ws=uW, bs=ub, act=O.TANH, env=env), dict(Ws=vW, bs=vb, act=O.TANH, env=env), X, None,
                                 -L, L, a=0.5, beta=X ** 2, E=E)
    m1, m2, m3, _ = m
    assert abs(m1 * m1 / (m2 + 1e-8) - g["loss_pde"]) <= TOL * max(1, abs(g["loss_pde"]))
    assert abs((2 * L * m3 - 1.0) ** 2 - g["loss_norm"]) <= TOL * max(1, abs(g["loss_norm"]))
    dtot = _wan_dtot(m1, m2, m3, 2 * L)
    assert_grads_close(stored_entries(_combine(Gu, dtot), g, "tot_u_"), grads_from(g, "tot_u_"), TOL, "tot/u")
    assert_grads_close(stored_entries(_combine(Gv, dtot), g, "tot_v_"), grads_from(g, "tot_v_"), TOL, "tot/v")
    assert abs(dtot[0] * dE1 - float(g["tot_gE"])) <= TOL * max(1, abs(float(g["tot_gE"])))


def test_reference_spread_is_recorded_for_every_fixture():
    """Every fixture carries the reference's own float32 run (ref32_*) and the conditioning of its float64
    outputs under one-ulp input changes (c64_*), which is what the GPU parity bars are derived from (conftest)."""
    import glob, os
    from conftest import GOLDEN
    worst = 0.0
    for f in sorted(glob.glob(os.path.join(GOLDEN, "*.npz"))):
        with np.load(f) as z:
            c = [k for k in z.files if k.startswith("c64_")]
            assert c and any(k.startswith("ref32_") for k in z.files) and any(k.startswith("e32_") for k in z.files), f
            for k in c:
                ref = np.max(np.abs(z[k[4:]]))
                if np.isfinite(z[k][0]) and ref > 0 and not k[4:].startswith(("u", "grad_u", "lap_u")):
                    worst = max(worst, z[k][0] / ref)
    # losses and gradient tensors: a one-ulp perturbation moves nothing by more than ~1e-12 relative to the tensor's
    # largest entry, so no float64 bar is loosened on conditioning grounds
    assert worst < 1e-12, worst


# ---------------------------------------------------------------- the flux, Ritz-value and parabolic programs
def _program_cases():
    """(program, d, bc, beta, f, faces) over d = 1..5 (parabolic 2..5), both envelopes, per-point and constant beta, f
    given and None; the flux program on one face, on all 2d faces and on a sparse mask of both ends of the face bits."""
    out = []
    for prog in ("flux", "ritz", "parabolic"):
        for d in range(2 if prog == "parabolic" else 1, 6):
            masks = {"one": 1 << (3 * d % (2 * d)), "all": (1 << 2 * d) - 1} if prog == "flux" else {"": 0}
            if prog == "flux" and d == 5:
                masks["sparse"] = 0b1000000001
            for bc in ("FBC", "RB"):
                for beta in ("point", "const"):
                    for f in ("f", "nof"):
                        for mname, faces in masks.items():
                            out.append(pytest.param(prog, d, bc, beta, f, faces,
                                                    id="-".join(x for x in (prog, f"d{d}", bc, beta, f, mname) if x)))
    return out


@pytest.mark.parametrize("prog,d,bc,beta,f,faces", _program_cases())
def test_numpy_programs_match_the_autograd_specifications(prog, d, bc, beta, f, faces):
    """oracle/jets_numpy's flux_program, ritz_value_program and parabolic_program through _loss_and_grads equal the
    float64 nested-autograd specifications the GPU suites are checked against (tests/flux_oracle, ritz_oracle,
    heat_oracle): the mean, every parameter gradient and, for the parabolic program, d mean / dE."""
    from flux_oracle import flux_loss
    from heat_oracle import parabolic_loss
    from ritz_oracle import ritz_value_loss
    rng = np.random.default_rng([("flux", "ritz", "parabolic").index(prog), d, bc == "FBC", beta == "point", f == "f", faces])
    L, H, act = 2.0, 10, (O.TANH if d % 2 else O.SIN)
    widths = [d, H, H, 1]
    Ws = [rng.uniform(-1, 1, (o, i)) / math.sqrt(i) for i, o in zip(widths[:-1], widths[1:])]
    bs = [rng.uniform(-0.5, 0.5, o) for o in widths[1:]]
    nf = bin(faces).count("1")
    N = 6 * nf if prog == "flux" else 23
    X = rng.uniform(0.1 * L, 0.9 * L, (N, d))
    if prog == "flux":      # the face coordinate of each block on its side of the box
        ax, s = O.face_blocks(faces, N)
        X[np.arange(N), ax] = np.where(s > 0, L, 0.0)
    bt = rng.uniform(0.5, 1.5, (N, 1)) if beta == "point" else 0.625
    fv = rng.normal(size=(N, 1)) if f == "f" else None
    alpha = {"flux": 0.75, "ritz": -1.25, "parabolic": -0.3}[prog]
    E = 0.375
    env = {"kind": O.ENV_POLY if bc == "FBC" else O.ENV_NONE, "lo": 0.0, "hi": L}
    order = {"flux": 1, "ritz": 0, "parabolic": 2}[prog]

    def program(U):
        dE = 0.0
        if prog == "flux":
            q, Ub = O.flux_program(U, d, faces, fv, alpha, bt)
        elif prog == "ritz":
            q, Ub = O.ritz_value_program(U, fv, alpha, bt)
        else:
            q, Ub, dE = O.parabolic_program(U, d, fv, alpha, bt, E)
        return float(q.mean()), Ub / N, dE / N

    loss, gWs, gbs, dE = O._loss_and_grads(Ws, bs, X, act, order, env, program)

    net = AR.build_mlp(widths, "tanh" if act == O.TANH else "sin", torch.float64)
    AR.load_params(net, Ws, bs)
    Xt = torch.tensor(X).requires_grad_(prog != "ritz")
    bt_t = torch.tensor(bt) if beta == "point" else bt
    f_t = None if fv is None else torch.tensor(fv)
    Et = torch.tensor(E, dtype=torch.float64, requires_grad=True)
    if prog == "flux":
        spec = flux_loss(net, Xt, faces, f_t, L, bc, alpha=alpha, kappa=bt_t)
    elif prog == "ritz":
        spec = ritz_value_loss(net, Xt, f_t, L, bc, kappa=bt_t, alpha=alpha)
    else:
        spec = parabolic_loss(net, Xt, f_t, alpha, bt_t, Et, L, bc)
    spec.backward()
    ps = [p.grad.numpy() for p in net.parameters()]
    tol = 1e-12
    assert abs(loss - float(spec.detach())) <= tol * max(1.0, abs(float(spec.detach()))), (loss, float(spec.detach()))
    assert_grads_close((gWs, gbs), (ps[0::2], ps[1::2]), tol, f"{prog} d{d} {bc}")
    if prog == "parabolic":
        assert abs(dE - float(Et.grad)) <= tol * max(1.0, abs(float(Et.grad))), (dE, float(Et.grad))
