"""Generate the golden fixtures in this directory from the LIVE reference.

Needs a checkout of the reference (its root in PDE_REFERENCE):
    python tests/golden/make_golden.py
The reference holds no golden vectors of its own (SURVEY.md §4), so these fixtures —
outputs of the reference's own loss functions and ``.backward()`` on seeded weights and
points, in float64 — are what pins ``oracle/`` and, through it, the CUDA path.
Nothing in ``tests/`` reads /root/reference at run time; only this script does.
"""
from __future__ import annotations

import copy
import importlib.util
import math
import os
import sys
import tempfile
import types

import numpy as np
import torch

REF = os.environ.get("PDE_REFERENCE", "/root/reference")
OUT = os.path.dirname(os.path.abspath(__file__))


def load_ref(relpath, name):
    """Import a reference script by path: stub matplotlib, run from a temp cwd
    (the Schrödinger scripts create results/ folders at import time)."""
    for m in ("matplotlib", "matplotlib.pyplot", "matplotlib.colors", "matplotlib.cm"):
        if m not in sys.modules:
            stub = types.ModuleType(m)
            sys.modules[m] = stub
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].use = lambda *a, **k: None
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp()
    os.chdir(tmp)
    try:
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, relpath))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        os.chdir(cwd)
    return mod


def linears(seq):
    return [m for m in seq if isinstance(m, torch.nn.Linear)]


def params_np(seq, prefix):
    d = {}
    for i, m in enumerate(linears(seq)):
        d[f"{prefix}W{i}"] = m.weight.detach().numpy().copy()
        d[f"{prefix}b{i}"] = m.bias.detach().numpy().copy()
    return d


def grads_np(seq, prefix):
    d = {}
    for i, m in enumerate(linears(seq)):
        gw = m.weight.grad
        gb = m.bias.grad
        d[f"{prefix}gW{i}"] = (torch.zeros_like(m.weight) if gw is None else gw).detach().numpy().copy()
        d[f"{prefix}gb{i}"] = (torch.zeros_like(m.bias) if gb is None else gb).detach().numpy().copy()
    return d


def zero_grads(*mods):
    for m in mods:
        for p in m.parameters():
            p.grad = None


# Keeps every fixture file under 1 MB: the config-5 networks have 200 x 200 and 100 x 100 hidden layers.
LARGE = 8192          # entries
SAMPLE = 2048


def shrink(arrs):
    """Arrays of more than LARGE entries, stored so that the tests compare exactly what they compared before or a fixed
    subset of it:
      - weights and biases that float32 represents exactly are stored as float32 (conftest.load_golden reads them back
        as float64, bit for bit);
      - an output gradient <key> keeps SAMPLE entries drawn with a fixed seed plus its largest-magnitude entry (so the
        max-abs scale of the comparison is unchanged), with their flat indices in <key>_idx; ref32_<key> keeps the same
        entries.  The norm in e32_<key>[1] and c64_<key>[1] is scaled by |sample| / |tensor| so that the relative-L2
        bar derived from it (conftest.grads_bar) is the full tensor's."""
    out = dict(arrs)
    for k, v in arrs.items():
        v = np.asarray(v)
        if v.size <= LARGE or k.startswith(("ref32_", "e32_", "c64_")):
            continue
        if "_g" not in k:
            if v.dtype == np.float64 and np.array_equal(v.astype(np.float32), v):
                out[k] = v.astype(np.float32)
            continue
        flat = v.reshape(-1)
        rng = np.random.default_rng(20240917)
        idx = np.union1d(rng.choice(flat.size, SAMPLE, replace=False), [int(np.argmax(np.abs(flat)))])
        idx = idx.astype(np.min_scalar_type(flat.size - 1))
        out[k], out[k + "_idx"] = flat[idx], idx
        if "ref32_" + k in arrs:
            out["ref32_" + k] = np.asarray(arrs["ref32_" + k]).reshape(-1)[idx]
        ratio = np.linalg.norm(flat[idx]) / np.linalg.norm(flat)
        for s in ("e32_", "c64_"):
            if s + k in arrs:
                out[s + k] = np.asarray(arrs[s + k], dtype=np.float64) * [1.0, ratio]
    return out


def save(name, **arrs):
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **shrink(arrs))
    print(f"wrote {name}.npz  ({os.path.getsize(path) / 1024:.0f} KiB)")


# ------------------------------------------------------------------ the reference's own numerical spread
# Every fixture also records how far the REFERENCE moves on the same case
#   ref32_<key> : the same reference code run in float32 (weights and points rounded to float32);
#   e32_<key>   : [max |ref32 - ref64|, ||ref32 - ref64||_2], worst case over the fixture itself and E32_DRAWS
#                 neighbouring inputs (every weight, bias and point moved by at most one float32 ulp, float64
#                 and float32 runs on the same moved inputs).  One draw is not enough: where two seeded gradient
#                 terms cancel (WAN critic biases) the reference's float32 error on a single input varies by two
#                 orders of magnitude.  The bar an fp32 implementation is held to is max(1e-5, 2 e32) relative;
#   c64_<key>   : [max |delta|, ||delta||_2] of the float64 result when every weight, bias and point is changed by
#                 at most one float64 ulp (three draws, worst case): the conditioning of that output.
# `compute(mods, T)` runs the reference on deep copies, so the float64 goldens themselves are untouched.
PERT_DRAWS = 3
E32_DRAWS = 8


def _np64(v):
    return np.asarray(v.detach().numpy() if torch.is_tensor(v) else v, dtype=np.float64)


def _perturbed(mods, T, gen, ulp):
    mp = {k: copy.deepcopy(m) for k, m in mods.items()}
    with torch.no_grad():
        for m in mp.values():
            for p in m.parameters():
                p.mul_(1.0 + (torch.rand(p.shape, generator=gen, dtype=torch.float64) * 2 - 1) * ulp)
    tp = {k: (v * (1.0 + (torch.rand(v.shape, generator=gen, dtype=torch.float64) * 2 - 1) * ulp)
              if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in T.items()}
    return mp, tp


def _as32(mods, T):
    return ({k: copy.deepcopy(m).float() for k, m in mods.items()},
            {k: (v.float() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in T.items()})


def _worse(worst, k, d):
    d = np.abs(d).reshape(-1)
    d = d[np.isfinite(d)] if np.isfinite(d).any() else d
    cur = np.array([d.max(), np.linalg.norm(d)])
    worst[k] = cur if worst.get(k) is None else np.maximum(worst[k], cur)


def reference_spread(mods, T, compute, base, skip=()):
    out = {}
    e32 = {}
    r32 = compute(*_as32(mods, T))
    for k, v in r32.items():
        if k not in skip:
            out["ref32_" + k] = np.asarray(_np64(v), dtype=np.float32)
            _worse(e32, k, _np64(v) - _np64(base[k]))
    gen = torch.Generator().manual_seed(987654321)
    c64 = {}
    for _ in range(PERT_DRAWS):
        mp, tp = _perturbed(mods, T, gen, 2.0 ** -52)
        for k, v in compute(mp, tp).items():
            if k not in skip:
                _worse(c64, k, _np64(v) - _np64(base[k]))
    gen = torch.Generator().manual_seed(123456789)
    for _ in range(E32_DRAWS):
        mp, tp = _perturbed(mods, T, gen, 2.0 ** -24)
        r64 = compute(mp, tp)
        r32 = compute(*_as32(mp, tp))
        for k in r64:
            if k not in skip:
                _worse(e32, k, _np64(r32[k]) - _np64(r64[k]))
    for k, v in c64.items():
        out["c64_" + k] = v
    for k, v in e32.items():
        out["e32_" + k] = v
    return out


# ------------------------------------------------------------------ Poisson
def emit(tag, mods, T, compute, meta, skip=()):
    """Run the reference (float64 = the golden values), then its float32 / perturbed-input spreads.
    `skip`: outputs not stored at all (per-point fields of the 40 000-point grids)."""
    base = compute(mods, T)
    extra = reference_spread(mods, T, compute, base, skip)
    save(tag, **meta, **{k: _np64(v) for k, v in base.items() if k not in skip}, **extra)


def with_prefix(prefix, d):
    return {prefix + k: v for k, v in d.items()}


def poisson_cases(P):
    L = 2.0
    # (tag, dim, width, depth, bc_mode, method, N)
    cases = [
        ("poisson_pinn_d1_w64_fbc", 1, 64, 5, "FBC", "pinn", 64),   # BASELINE config 1 shape
        ("poisson_pinn_d3_w64_fbc", 3, 64, 5, "FBC", "pinn", 64),   # BASELINE config 2 shape
        ("poisson_drm_d5_w64_rb", 5, 64, 5, "RB", "drm", 64),       # BASELINE config 3 shape
        ("poisson_pinn_d2_w16_fbc", 2, 16, 4, "FBC", "pinn", 96),
        ("poisson_pinn_d5_w16_fbc", 5, 16, 3, "FBC", "pinn", 96),
        ("poisson_pinn_d3_w16_rb", 3, 16, 4, "RB", "pinn", 96),
        ("poisson_pinn_d4_w12_fbc", 4, 12, 3, "FBC", "pinn", 50),   # ragged width / N
        ("poisson_drm_d1_w16_fbc", 1, 16, 4, "FBC", "drm", 96),
        ("poisson_drm_d2_w16_fbc", 2, 16, 4, "FBC", "drm", 96),
        ("poisson_drm_d3_w16_fbc", 3, 16, 4, "FBC", "drm", 96),
    ]
    for k, (tag, d, w, depth, bc, method, N) in enumerate(cases):
        torch.manual_seed(100 + k)
        model = P.SolutionNet(d, w, depth, bc_mode=bc).double()
        X = (torch.rand(N, d, dtype=torch.float64) * L).requires_grad_(True)
        ks = [1 + (i % 2) for i in range(d)]
        f = P.rhs_f_for_u_sin(X, L, ks).detach()
        fn = P.pinn_residual_loss if method == "pinn" else P.drm_energy_loss

        def compute(mods, T, fn=fn):
            model = mods["u"]
            X = T["X"].clone().requires_grad_(True)
            zero_grads(model)
            loss = fn(model, X, T["f"], L)
            loss.backward()
            # also the raw network jets the reference's helpers produce (u, grad u, laplacian)
            X2 = T["X"].clone().requires_grad_(True)
            u = model(X2, L)
            g = P.grad_scalar_field(u, X2)
            lap = P.laplacian(u, X2)
            return dict(loss=np.float64(loss.item()), u=u.detach().numpy(), grad_u=g.detach().numpy(),
                        lap_u=lap.detach().numpy(), **grads_np(model.net, ""))
        emit(tag, {"u": model}, {"X": X.detach(), "f": f}, compute,
             dict(X=X.detach().numpy(), f=f.numpy(), L=np.float64(L), **params_np(model.net, "")))

    # survey sanity pins (SURVEY.md §8c): default dtype float64, seed 0, model first, then X = rand(512,d)*2
    pins = {}
    torch.set_default_dtype(torch.float64)
    for d in (1, 2, 3, 5):
        torch.manual_seed(0)
        m = P.SolutionNet(d, 64, 5, "FBC").double()
        X = (torch.rand(512, d) * 2.0).requires_grad_(True)
        f = P.rhs_f_for_u_sin(X, 2.0, [1] * d).detach()
        pins[f"pinn_d{d}"] = P.pinn_residual_loss(m, X, f, 2.0).item()
        pins[f"drm_d{d}"] = P.drm_energy_loss(m, X, f, 2.0).item()
    expect = {"pinn_d1": 3.997824334710243, "pinn_d2": 6.755232513291217, "pinn_d3": 6.414617763140292,
              "pinn_d5": 4.878397382574168, "drm_d1": 0.2063688668551195, "drm_d2": 0.0828105207704522,
              "drm_d3": -0.04937656836661489, "drm_d5": 1.869090502863647e-4}
    torch.set_default_dtype(torch.float32)
    for k, v in expect.items():
        assert abs(pins[k] - v) <= 1e-12 * max(1.0, abs(v)), (k, pins[k], v)
    print("survey sanity pins reproduced:", {k: float(f"{v:.6g}") for k, v in pins.items()})

    # WAN (two networks), d=2
    torch.manual_seed(200)
    um = P.SolutionNet(2, 16, 4, bc_mode="FBC").double()
    vm = P.CriticNet(2, 16, 3).double()
    N = 96
    X = (torch.rand(N, 2, dtype=torch.float64) * L).requires_grad_(True)
    f = P.rhs_f_for_u_sin(X, L, [1, 2]).detach()
    poisson_wan_case(P, "poisson_wan_d2_w16", um, vm, X.detach(), f, L, 1.0)

    # the value-only terms of the epoch (Poisson_ND.py:130-147,230-239): data MSE, norm term, and the Dirichlet
    # face penalty on fixed face points (the reference draws them from the global RNG inside the function; the
    # fixture stores the draw so that every implementation sees the same points)
    torch.manual_seed(210)
    model = P.SolutionNet(3, 16, 4, bc_mode="RB").double()
    Xd = torch.rand(80, 3, dtype=torch.float64) * L
    ud = P.exact_u_prod_sin(Xd, L, [1, 2, 1]) + 0.05 * torch.randn(80, 1, dtype=torch.float64)
    Nb = 24
    faces = []
    for i in range(3):
        for val in (0.0, L):
            Xb = torch.rand(Nb, 3, dtype=torch.float64) * L
            Xb[:, i] = val
            faces.append(Xb)
    Xb_all = torch.stack(faces)      # (2d, Nb, d) in the order boundary_loss_dirichlet visits the faces

    def compute(mods, T):
        model = mods["u"]
        out = {}
        zero_grads(model)
        u = model(T["Xd"], L)
        ld = torch.mean((u - T["ud"]) ** 2)              # Poisson_ND.py:230-232
        ld.backward()
        out["data_loss"] = np.float64(ld.item()); out.update(grads_np(model.net, "data_"))
        for mode in ("nontrivial", "l2"):
            zero_grads(model)
            ln = P.norm_loss(model(T["Xd"], L), mode=mode)   # :143-147, :236-239
            ln.backward()
            out[f"norm_{mode}_loss"] = np.float64(ln.item()); out.update(grads_np(model.net, f"norm_{mode}_"))
        zero_grads(model)
        lb = sum(torch.mean(model(xb, L) ** 2) for xb in T["Xb"]) / T["Xb"].shape[0]    # :130-141 on the stored faces
        lb.backward()
        out["bc_loss"] = np.float64(lb.item()); out.update(grads_np(model.net, "bc_"))
        return out
    emit("poisson_value_terms_d3_w16_rb", {"u": model}, {"Xd": Xd, "ud": ud, "Xb": Xb_all}, compute,
         dict(Xd=Xd.numpy(), ud=ud.numpy(), Xb=Xb_all.numpy(), L=np.float64(L), **params_np(model.net, "")))


def poisson_wan_case(P, tag, um, vm, X, f, L, reg):
    def compute(mods, T):
        um, vm = mods["u"], mods["v"]
        X = T["X"].clone().requires_grad_(True)
        out = {}
        zero_grads(um, vm)
        lu, lv, weak, pn = P.wan_losses(um, vm, X, T["f"], L, v_reg_weight=reg)
        lu.backward(retain_graph=True)
        out.update(with_prefix("lu_", grads_np(um.net, "u_")))
        out.update(with_prefix("lu_", grads_np(vm.net, "v_")))
        zero_grads(um, vm)
        lv.backward()
        out.update(with_prefix("lv_", grads_np(um.net, "u_")))
        out.update(with_prefix("lv_", grads_np(vm.net, "v_")))
        out.update(loss_u=np.float64(lu.item()), loss_v=np.float64(lv.item()), weak=np.float64(weak.item()),
                   phi_norm=np.float64(pn.item()))
        return out
    emit(tag, {"u": um, "v": vm}, {"X": X, "f": f}, compute,
         dict(X=X.numpy(), f=f.numpy(), L=np.float64(L), v_reg_weight=np.float64(reg),
              **params_np(um.net, "u_"), **params_np(vm.net, "v_")))


# ------------------------------------------------------------------ 1-D well
def two_net_wan_outputs(loss_fn, um, vm, u_seq, v_seq, energy=None):
    """(total, loss_v, loss_pde, loss_norm) of a Schrödinger WAN_loss and the gradients of `total` and `loss_v`."""
    out = {}
    zero_grads(um, vm)
    total, lv, lpde, lnorm = loss_fn()
    total.backward(retain_graph=True)
    out.update(with_prefix("tot_", grads_np(u_seq, "u_")))
    out.update(with_prefix("tot_", grads_np(v_seq, "v_")))
    if energy is not None:
        out["tot_gE"] = energy.grad.numpy().copy()
    zero_grads(um, vm)
    lv.backward()
    out.update(with_prefix("lv_", grads_np(u_seq, "u_")))
    out.update(with_prefix("lv_", grads_np(v_seq, "v_")))
    if energy is not None:
        out["lv_gE"] = energy.grad.numpy().copy()
    out.update(total=np.float64(total.item()), loss_v=np.float64(lv.item()), loss_pde=np.float64(lpde.item()),
               loss_norm=np.float64(lnorm.item()))
    return out


def ipw_pinn_drm_case(I, tag, model, x, n, L):
    def compute(mods, T):
        model = mods["u"]
        x = T["x"].clone().requires_grad_(True)
        zero_grads(model)
        lp = I.PINN_loss(model, x, n, L)
        lp.backward()
        gp = grads_np(model.net, "pinn_")
        zero_grads(model)
        ld = I.DRM_loss(model, x)
        ld.backward()
        gd = grads_np(model.net, "drm_")
        return dict(pinn_loss=np.float64(lp.item()), drm_loss=np.float64(ld.item()), **gp, **gd)
    emit(tag, {"u": model}, {"x": x}, compute,
         dict(x=x.numpy(), L=np.float64(L), n=np.int64(n), **params_np(model.net, "")))


def ipw_wan_case(W, tag, um, vm, x, n, L):
    def compute(mods, T):
        um, vm = mods["u"], mods["v"]
        x = T["x"].clone().requires_grad_(True)
        return two_net_wan_outputs(lambda: W.WAN_loss(um, vm, x, n, L, 1.0, 1.0), um, vm, um.net, vm.net)
    emit(tag, {"u": um, "v": vm}, {"x": x}, compute,
         dict(x=x.numpy(), L=np.float64(L), n=np.int64(n), **params_np(um.net, "u_"), **params_np(vm.net, "v_")))


def ipw_cases(I, W):
    L = 2.0
    for tag, kw, n in (("ipw1d_fbc_n2", dict(enforce_bc=True), 2), ("ipw1d_fn_n3", dict(FN=True, num_states=3), 3)):
        torch.manual_seed(300 + n)
        model = I.FCN([1, 20, 20, 1], L=L, **kw).double()
        with torch.no_grad():      # reference zero-initialises biases; perturb so bias paths are exercised
            for m in linears(model.net):
                m.bias.uniform_(-0.3, 0.3)
        x = torch.linspace(0.0, L, 65, dtype=torch.float64).view(-1, 1)
        ipw_pinn_drm_case(I, tag, model, x, n, L)

    torch.manual_seed(310)
    um = W.FCN([1, 20, 20, 1], L=L, enforce_bc=True).double()
    vm = W.FCN([1, 10, 10, 1], L=L, enforce_bc=False).double()
    with torch.no_grad():
        for m in linears(um.net) + linears(vm.net):
            m.bias.uniform_(-0.3, 0.3)
    x = torch.linspace(0.0, L, 65, dtype=torch.float64).view(-1, 1)
    ipw_wan_case(W, "ipw1d_wan_n2", um, vm, x, 2, L)


# ------------------------------------------------------------------ 2-D oscillator
def grid2d(lo, hi, n, dtype=torch.float64):
    g1 = torch.linspace(lo, hi, n, dtype=dtype)
    xg, yg = torch.meshgrid(g1, g1, indexing="ij")
    return xg.clone(), yg.clone()


def qho2d_pinn_drm_case(Q, tag, model, x, y, nx, ny, L, store_grid=True):
    E = Q.Exact_energy(nx, ny, L)

    def compute(mods, T):
        model = mods["u"]
        x = T["x"].clone().requires_grad_(True)
        y = T["y"].clone().requires_grad_(True)
        # --- restatement of the inline residual block, QHO_2D.py:329-341,363-383 ---
        def jets():
            u = model(x, y)
            ux = torch.autograd.grad(u, x, torch.ones_like(u), create_graph=True)[0]
            uy = torch.autograd.grad(u, y, torch.ones_like(u), create_graph=True)[0]
            return u, ux, uy
        zero_grads(model)
        u, ux, uy = jets()
        V = 0.5 * math.sqrt(2) ** 2 * (x ** 2 + y ** 2)
        uxx = torch.autograd.grad(ux, x, torch.ones_like(ux), create_graph=True)[0]
        uyy = torch.autograd.grad(uy, y, torch.ones_like(uy), create_graph=True)[0]
        res = -0.5 * (uxx + uyy) + V * u - E * u
        lp = torch.mean(res ** 2)
        lp.backward()
        gp = grads_np(model.net, "pinn_")
        zero_grads(model)
        u, ux, uy = jets()
        V = 0.5 * math.sqrt(2) ** 2 * (x ** 2 + y ** 2)
        ld = torch.mean(0.5 * (ux ** 2 + uy ** 2) + V * u ** 2) / torch.mean(u ** 2 + 1e-8)
        ld.backward()
        gd = grads_np(model.net, "drm_")
        return dict(pinn_loss=np.float64(lp.item()), drm_loss=np.float64(ld.item()), u=u.detach().numpy(), **gp, **gd)
    grid = dict(x=x.numpy(), y=y.numpy()) if store_grid else dict(grid_n=np.int64(x.shape[0]))
    emit(tag, {"u": model}, {"x": x, "y": y}, compute,
         dict(L=np.float64(L), nx=np.int64(nx), ny=np.int64(ny), E=np.float64(E), nodes_x=model.nodes_x.double().numpy(),
              nodes_y=model.nodes_y.double().numpy(), **grid, **params_np(model.net, "")),
         skip=() if store_grid else ("u",))


def qho2d_wan_case(Q, tag, um, vm, x, y, nx, ny, L, store_grid=True):
    def compute(mods, T):
        um, vm = mods["u"], mods["v"]
        x = T["x"].clone().requires_grad_(True)
        y = T["y"].clone().requires_grad_(True)
        return two_net_wan_outputs(lambda: Q.WAN_loss(um, vm, x, y, nx, ny, L, 1.0, 1.0), um, vm, um.net, vm.net)
    grid = dict(x=x.numpy(), y=y.numpy()) if store_grid else dict(grid_n=np.int64(x.shape[0]))
    emit(tag, {"u": um, "v": vm}, {"x": x, "y": y}, compute,
         dict(L=np.float64(L), nx=np.int64(nx), ny=np.int64(ny), E=np.float64(Q.Exact_energy(nx, ny, L)), **grid,
              **params_np(um.net, "u_"), **params_np(vm.net, "v_")))


def qho2d_cases(Q):
    L = 6.0
    for tag, tech, nx, ny in (("qho2d_fbc_00", "FBC", 0, 0), ("qho2d_fn_21", "FN", 2, 1)):
        torch.manual_seed(400 + nx)
        model = Q.FCN([2, 16, 16, 16, 1], nx, ny, tech).double()
        x, y = grid2d(-L, L, 12)
        qho2d_pinn_drm_case(Q, tag, model, x, y, nx, ny, L)

    torch.manual_seed(410)
    nx, ny = 1, 0
    um = Q.FCN([2, 16, 16, 1], nx, ny, "FBC").double()
    vm = Q.FCN([2, 10, 10, 1], nx, ny, "FBC").double()
    x, y = grid2d(-L, L, 12)
    qho2d_wan_case(Q, "qho2d_wan_10", um, vm, x, y, nx, ny, L)


# ------------------------------------------------------------------ Kramers–Henneberger
def kh_case(K, tag, model, vm, x, L, alpha, V0, wan_model=None):
    """PINN / DRM on `model`; WAN on `wan_model` (defaults to `model`) with critic `vm`."""
    mods = {"u": model, "v": vm}
    if wan_model is not None:
        mods["w"] = wan_model

    def compute(mods, T):
        model, vm = mods["u"], mods["v"]
        wm = mods.get("w", model)
        x = T["x"].clone().requires_grad_(True)
        out = {}
        zero_grads(model, vm, wm)
        lp = K.pinn_loss(model, x, alpha, V0)
        lp.backward()
        out.update(grads_np(model.u_model.net, "pinn_")); out["pinn_gE"] = model.energy.grad.numpy().copy()
        zero_grads(model, vm, wm)
        ld = K.drm_loss(model, x, alpha, V0, L)
        ld.backward()
        out.update(grads_np(model.u_model.net, "drm_"))
        zero_grads(model, vm, wm)
        lw, ln = K.wan_loss(wm, vm, x, alpha, V0, L)
        (lw + ln).backward()
        out.update(grads_np(wm.u_model.net, "wan_u_")); out.update(grads_np(vm.net, "wan_v_"))
        out["wan_gE"] = wm.energy.grad.numpy().copy()
        out.update(pinn_loss=np.float64(lp.item()), drm_loss=np.float64(ld.item()), wan_pde=np.float64(lw.item()),
                   wan_norm=np.float64(ln.item()))
        return out
    Vx = K.V_KH(x, alpha=alpha, V0=V0, use_avg=True, n_theta=500)
    meta = dict(x=x.numpy(), V=Vx.numpy(), L=np.float64(L), alpha=np.float64(alpha), E=np.float64(model.energy.item()),
                **params_np(model.u_model.net, "u_"), **params_np(vm.net, "v_"))
    if wan_model is not None:
        meta.update(params_np(wan_model.u_model.net, "w_"))
    emit(tag, mods, {"x": x}, compute, meta)


def kh_cases(K):
    L, alpha, V0 = 12.0, 2.0, -24.856
    for tag, tech in (("kh1d_raw", "RAW"), ("kh1d_fbc", "FBC")):
        torch.manual_seed(500)
        model = K.UnifiedEigenModel([1, 16, 16, 1], technique=tech, E_init=-3.0, device="cpu").double()
        vm = K.FCN1D([1, 10, 10, 1], technique="RAW").double()
        x = torch.linspace(-L, L, 96, dtype=torch.float64)
        kh_case(K, tag, model, vm, x, L, alpha, V0)


# ------------------------------------------------------------------ remaining Schrödinger scripts
def perturb_biases(*seqs):
    with torch.no_grad():
        for seq in seqs:
            for m in seq:
                if isinstance(m, torch.nn.Linear):
                    m.bias.uniform_(-0.3, 0.3)


def qho1d_wan_case(QW, tag, um, vm, x, n, L):
    def compute(mods, T):
        um, vm = mods["u"], mods["v"]
        x = T["x"].clone().requires_grad_(True)
        return two_net_wan_outputs(lambda: QW.WAN_loss(um, vm, x, n, L, 1.0, 1.0), um, vm, um.net, vm.net, um.energies)
    emit(tag, {"u": um, "v": vm}, {"x": x}, compute,
         dict(x=x.numpy(), L=np.float64(L), n=np.int64(n), E=np.float64(um.energies.item()),
              **params_np(um.net, "u_"), **params_np(vm.net, "v_")))


def qho1d_cases(Q1, QW):
    """QHO_1D_PINN_DRM.py (ModuleList sine network, exp-window / forced nodes) and QHO_1D_WAN.py
    (tanh networks, trainable energies)."""
    X_max = 6.0
    for tag, n, kw in (("qho1d_bc_n1", 1, dict(enforce_bc=True)), ("qho1d_fn_n2", 2, dict(enforce_bc=True, FN=True)),
                       ("qho1d_fnonly_n3", 3, dict(enforce_bc=False, FN=True))):
        torch.manual_seed(600 + n)
        model = Q1.FCN_Single([1, 20, 20, 1], num_states=n, domain_length=2 * X_max, **kw).double()
        x = torch.linspace(-X_max, X_max, 81, dtype=torch.float64).view(-1, 1)

        def compute(mods, T, n=n):
            model = mods["u"]
            x = T["x"].clone().requires_grad_(True)
            out = {}
            for nm, fn in (("pinn", lambda: Q1.PINN_loss(model, x)), ("drm", lambda: Q1.DRM_loss(model, x)),
                           ("norm", lambda: Q1.normalization_loss(model, x)),
                           ("orth", lambda: Q1.Orthogonal_loss(model, x, n, X_max))):
                zero_grads(model)
                l = fn()
                l.backward()
                out[nm + "_loss"] = np.float64(l.item())
                out.update(grads_np(model.net.layers, nm + "_"))
            return out
        emit(tag, {"u": model}, {"x": x}, compute,
             dict(x=x.numpy(), X_max=np.float64(X_max), n=np.int64(n), **params_np(model.net.layers, "")))

    torch.manual_seed(620)
    L, n = 6.0, 1
    um = QW.FCN([1, 20, 20, 1], num_states=n, L=L, enforce_bc=True).double()
    vm = QW.FCN([1, 10, 10, 1], num_states=n, L=L, enforce_bc=False).double()
    perturb_biases(um.net, vm.net)
    with torch.no_grad():
        um.energies.add_(0.1)
    x = torch.linspace(-L, L, 81, dtype=torch.float64).view(-1, 1)
    qho1d_wan_case(QW, "qho1d_wan_n1", um, vm, x, n, L)


def ipw_fn_wan_case(WF):
    """IPW_1D_WAN_FN.py: forced-node ansatz on both networks."""
    torch.manual_seed(630)
    L, n = 2.0, 3
    um = WF.FCN([1, 20, 20, 1], num_states=n, L=L).double()
    vm = WF.FCN([1, 10, 10, 1], num_states=1, L=L).double()
    perturb_biases(um.net, vm.net)
    x = torch.linspace(0.0, L, 65, dtype=torch.float64).view(-1, 1)
    ipw_wan_case(WF, "ipw1d_wanfn_n3", um, vm, x, n, L)


def ipw2d_case(I2, tag, model, x, y, nx, ny, L, store_grid=True):
    k2 = (2 * ((nx * np.pi) ** 2 / (2 * L ** 2) + (ny * np.pi) ** 2 / (2 * L ** 2)))

    def compute(mods, T):
        model = mods["u"]
        x = T["x"].clone().requires_grad_(True)
        y = T["y"].clone().requires_grad_(True)

        def jets():
            u = model(x, y)
            ux = torch.autograd.grad(u, x, torch.ones_like(u), create_graph=True)[0]
            uy = torch.autograd.grad(u, y, torch.ones_like(u), create_graph=True)[0]
            return u, ux, uy
        zero_grads(model)
        u, ux, uy = jets()
        uxx = torch.autograd.grad(ux, x, torch.ones_like(ux), create_graph=True)[0]
        uyy = torch.autograd.grad(uy, y, torch.ones_like(uy), create_graph=True)[0]
        lp = torch.mean((uxx + uyy + k2 * u) ** 2)
        lp.backward()
        gp = grads_np(model.net, "pinn_")
        zero_grads(model)
        u, ux, uy = jets()
        ld = torch.mean(ux ** 2 + uy ** 2) / torch.mean(u ** 2 + 1e-8)
        ld.backward()
        gd = grads_np(model.net, "drm_")
        zero_grads(model)
        lo = I2.orthogonal_loss(model, x, y, nx, ny, L)
        go = {}
        if torch.is_tensor(lo) and lo.requires_grad:
            lo.backward()
            go = grads_np(model.net, "orth_")
        return dict(pinn_loss=np.float64(lp.item()), drm_loss=np.float64(ld.item()), orth_loss=np.float64(float(lo)),
                    u=u.detach().numpy(), **gp, **gd, **go)
    grid = dict(x=x.numpy(), y=y.numpy()) if store_grid else dict(grid_n=np.int64(x.shape[0]))
    emit(tag, {"u": model}, {"x": x, "y": y}, compute,
         dict(L=np.float64(L), nx=np.int64(nx), ny=np.int64(ny), **grid, **params_np(model.net, "")),
         skip=() if store_grid else ("u",))


def ipw2d_cases(I2):
    """IPW_2D.py: the inline PINN / DRM blocks of train_pinn_seperate (:195-228) restated around the
    imported FCN, plus orthogonal_loss (:113-126)."""
    L = 2.0
    for tag, tech, nx, ny in (("ipw2d_fbc_11", "FBC", 1, 1), ("ipw2d_fn_32", "FN", 3, 2)):
        torch.manual_seed(640 + nx)
        model = I2.FCN([2, 16, 16, 16, 1], nx, ny, tech).double()
        x, y = grid2d(0.0, L, 12)
        ipw2d_case(I2, tag, model, x, y, nx, ny, L)


def qho2d_energy_case(QE):
    """QHO_2D_Energy.py: PINN residual with the trainable energy E_train (:287-291,382-383)."""
    L, nx, ny = 6.0, 1, 1
    torch.manual_seed(650)
    model = QE.FCN([2, 16, 16, 16, 1], nx, ny, "FBC").double()
    E_holder = torch.nn.Module()
    E_holder.E = torch.nn.Parameter(torch.tensor(QE.Exact_energy(nx, ny, L) + 0.05, dtype=torch.float64))
    x, y = grid2d(-L, L, 12)

    def compute(mods, T):
        model, E_train = mods["u"], mods["E"].E
        x = T["x"].clone().requires_grad_(True)
        y = T["y"].clone().requires_grad_(True)
        u = model(x, y)
        ux = torch.autograd.grad(u, x, torch.ones_like(u), create_graph=True)[0]
        uy = torch.autograd.grad(u, y, torch.ones_like(u), create_graph=True)[0]
        uxx = torch.autograd.grad(ux, x, torch.ones_like(ux), create_graph=True)[0]
        uyy = torch.autograd.grad(uy, y, torch.ones_like(uy), create_graph=True)[0]
        V = 0.5 * math.sqrt(2) ** 2 * (x ** 2 + y ** 2)
        lp = torch.mean((-0.5 * (uxx + uyy) + V * u - E_train * u) ** 2)
        zero_grads(model, mods["E"])
        lp.backward()
        return dict(pinn_loss=np.float64(lp.item()), pinn_gE=E_train.grad.numpy().copy(), **grads_np(model.net, "pinn_"))
    emit("qho2d_energy_11", {"u": model, "E": E_holder}, {"x": x, "y": y}, compute,
         dict(x=x.numpy(), y=y.numpy(), L=np.float64(L), nx=np.int64(nx), ny=np.int64(ny), E=np.float64(E_holder.E.item()),
              **params_np(model.net, "")))


# ------------------------------------------------------------------ BASELINE.json configs 4 and 5 at their own shapes
def config_shaped(Q, I2, W, K, QW):
    """Networks, grids and constants of the reference's own __main__ blocks (QHO_2D.py:249-254,281-282;
    IPW_2D.py:137-138,166; IPW_1D_WAN.py:140-141,163-166; KH_1D.py:624-638,307-310,331-335; QHO_1D_WAN.py:159,169-176).
    Default initialisation; zero-initialised biases are perturbed so the bias paths carry signal."""
    # config 4: 2-D eigenstate PINN / Rayleigh on the 200 x 200 grid (end points included)
    L = 6.0
    for tag, tech, nx, ny in (("cfg4_qho2d_fbc_00", "FBC", 0, 0), ("cfg4_qho2d_fn_21", "FN", 2, 1)):
        torch.manual_seed(700 + nx)
        model = Q.FCN([2, 50, 50, 50, 50, 1], nx, ny, tech).double()
        x, y = grid2d(-L, L, 200)
        qho2d_pinn_drm_case(Q, tag, model, x, y, nx, ny, L, store_grid=False)
    torch.manual_seed(710)
    um = Q.FCN([2, 50, 50, 50, 50, 1], 1, 0, "FBC").double()
    vm = Q.FCN([2, 20, 20, 20, 1], 1, 0, "FBC").double()
    x, y = grid2d(-L, L, 200)
    qho2d_wan_case(Q, "cfg4_qho2d_wan_10", um, vm, x, y, 1, 0, L, store_grid=False)
    L = 2.0
    for tag, tech, nx, ny in (("cfg4_ipw2d_fbc_11", "FBC", 1, 1), ("cfg4_ipw2d_fn_32", "FN", 3, 2)):
        torch.manual_seed(720 + nx)
        model = I2.FCN([2, 50, 50, 50, 50, 1], nx, ny, tech).double()
        x, y = grid2d(0.0, L, 200)
        ipw2d_case(I2, tag, model, x, y, nx, ny, L, store_grid=False)

    # config 5: WAN minimax pairs
    torch.manual_seed(730)
    L, n = 2.0, 2
    um = W.FCN([1, 50, 50, 50, 1], num_states=n, L=L, enforce_bc=True).double()
    vm = W.FCN([1, 20, 20, 20, 1], num_states=n, L=L, enforce_bc=False).double()
    perturb_biases(um.net, vm.net)
    x = torch.linspace(0.0, L, 1000, dtype=torch.float64).view(-1, 1)
    ipw_wan_case(W, "cfg5_ipw1d_wan_n2", um, vm, x, n, L)

    torch.manual_seed(740)
    L, alpha, V0 = 60.0, 10.0, -24.856
    model = K.UnifiedEigenModel([1, 100, 100, 100, 1], technique="FBC", E_init=-1.2, device="cpu").double()   # PINN / DRM
    wmodel = K.UnifiedEigenModel([1, 100, 100, 100, 1], technique="RAW", E_init=-1.2, device="cpu").double()  # WAN (:331)
    vm = K.FCN1D([1, 50, 50, 50, 1], technique="RAW").double()
    x = torch.linspace(-L, L, 1024, dtype=torch.float64)
    kh_case(K, "cfg5_kh1d_a10", model, vm, x, L, alpha, V0, wan_model=wmodel)

    torch.manual_seed(750)
    L, n = 6.0, 1
    um = QW.FCN([1, 200, 200, 200, 1], num_states=n, L=L, enforce_bc=True).double()
    vm = QW.FCN([1, 100, 100, 100, 1], num_states=n, L=L, enforce_bc=True).double()
    perturb_biases(um.net, vm.net)
    x = torch.linspace(-L, L, 1000, dtype=torch.float64).view(-1, 1)
    qho1d_wan_case(QW, "cfg5_qho1d_wan_n1", um, vm, x, n, L)


def main():
    torch.set_default_dtype(torch.float32)
    P = load_ref("Poisson_Equations/Poisson_ND.py", "ref_poisson_nd")
    poisson_cases(P)
    I = load_ref("Schrodinger_Equations/Infinite_Potential_Well/IPW_1D_PINN_DRM.py", "ref_ipw_pd")
    W = load_ref("Schrodinger_Equations/Infinite_Potential_Well/IPW_1D_WAN.py", "ref_ipw_wan")
    ipw_cases(I, W)
    Q = load_ref("Schrodinger_Equations/Quantum_Harmonic_Oscillator/QHO_2D.py", "ref_qho2d")
    qho2d_cases(Q)
    K = load_ref("Schrodinger_Equations/Kramers_Henneberger/KH_1D.py", "ref_kh1d")
    kh_cases(K)
    more()
    configs()


def more():
    """The scripts added after the first fixture set (run alone with ``make_golden.py more``)."""
    torch.set_default_dtype(torch.float32)
    Q1 = load_ref("Schrodinger_Equations/Quantum_Harmonic_Oscillator/QHO_1D_PINN_DRM.py", "ref_qho1d_pd")
    QW = load_ref("Schrodinger_Equations/Quantum_Harmonic_Oscillator/QHO_1D_WAN.py", "ref_qho1d_wan")
    qho1d_cases(Q1, QW)
    WF = load_ref("Schrodinger_Equations/Infinite_Potential_Well/IPW_1D_WAN_FN.py", "ref_ipw_wanfn")
    ipw_fn_wan_case(WF)
    I2 = load_ref("Schrodinger_Equations/Infinite_Potential_Well/IPW_2D.py", "ref_ipw2d")
    ipw2d_cases(I2)
    QE = load_ref("Schrodinger_Equations/Quantum_Harmonic_Oscillator/QHO_2D_Energy.py", "ref_qho2d_energy")
    qho2d_energy_case(QE)


def configs():
    """Fixtures at the shapes BASELINE.json configs 4 and 5 name (run alone with ``make_golden.py configs``)."""
    torch.set_default_dtype(torch.float32)
    Q = load_ref("Schrodinger_Equations/Quantum_Harmonic_Oscillator/QHO_2D.py", "ref_qho2d")
    I2 = load_ref("Schrodinger_Equations/Infinite_Potential_Well/IPW_2D.py", "ref_ipw2d")
    W = load_ref("Schrodinger_Equations/Infinite_Potential_Well/IPW_1D_WAN.py", "ref_ipw_wan")
    K = load_ref("Schrodinger_Equations/Kramers_Henneberger/KH_1D.py", "ref_kh1d")
    QW = load_ref("Schrodinger_Equations/Quantum_Harmonic_Oscillator/QHO_1D_WAN.py", "ref_qho1d_wan")
    config_shaped(Q, I2, W, K, QW)


if __name__ == "__main__":
    {"more": more, "configs": configs}.get((sys.argv[1:] or [""])[0], main)()
