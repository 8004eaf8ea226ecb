"""GPU tests of Deep Ritz with Neumann / Robin data: the Ritz value program (PDE_PROG_RITZ_VALUE) on both kernel families
against the float64 autograd specification (tests/ritz_oracle.py), the Poisson drop-ins boundary_energy_neumann and
mean_value_loss, FusedTrainer's Ritz boundary term, Robin data and mean constraint against a reference-style loop, the
folded multi-GPU exchange, and the convergence bound of case (a) of tools/ritz_convergence.py.

Bars (DESIGN.md §7): float64 on the generic kernel 1e-10; float32 max(1e-5, 2 e32), e32 being the distance between the
specification run in float32 and in float64 on the same inputs (and on inputs one float32 ulp away)."""
import copy
import os
import socket
import sys

import numpy as np
import pytest
import torch

from conftest import grads_err
from flux_oracle import flux_loss
from ritz_oracle import boundary_energy, exact_mean, mean_value_loss, ritz_energy, ritz_value_loss
from test_gpu_neumann import _f32, _g_autograd, _grads, _Holder, _net

pytestmark = pytest.mark.gpu
L_BOX = 2.0


def _oracle(net, X, g, bc, alpha, kappa, dtype=torch.float64):
    """(loss, grads) of the specification on the CPU in ``dtype``."""
    ref = copy.deepcopy(net).to(dtype)
    Xt = torch.tensor(X, dtype=dtype)
    gt = None if g is None else torch.tensor(g, dtype=dtype)
    kt = torch.tensor(kappa, dtype=dtype) if isinstance(kappa, np.ndarray) else kappa
    loss = ritz_value_loss(ref, Xt, gt, L_BOX, bc, kappa=kt, alpha=alpha)
    loss.backward()
    return float(loss.detach()), _grads(ref)


def _e32(net, X, g, bc, alpha, kappa, draws=8):
    """The specification's own float32 error: the worst case over these inputs and eight inputs one float32 ulp away
    (the rule of test_gpu_neumann.py)."""
    gen = np.random.default_rng(7)
    worst = 0.0
    for k in range(draws + 1):
        jit = (lambda t: t * (1.0 + gen.uniform(-1, 1, t.shape) * 2.0 ** -24)) if k else (lambda t: t)
        netj = copy.deepcopy(net)
        if k:
            with torch.no_grad():
                for p in netj.parameters():
                    p.copy_(torch.tensor(jit(p.detach().numpy())))
        Xj, gj = jit(X), None if g is None else jit(g)
        kj = jit(kappa) if isinstance(kappa, np.ndarray) else kappa
        l32, g32 = _oracle(netj, Xj, gj, bc, alpha, kj, torch.float32)
        l64, g64 = _oracle(netj, Xj, gj, bc, alpha, kj, torch.float64)
        worst = max(worst, abs(l32 - l64) / max(abs(l64), 1e-3), grads_err(g32, g64)[0])
    return worst


def _kernel(net, X, g, bc, alpha, kappa, dtype, path):
    """loss and gradients of the RITZ_VALUE program through ops.residual_means on the given kernel family."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import EnvelopeSpec, ProgramSpec, NO_ENVELOPE, residual_means
    m = copy.deepcopy(net).to("cuda", dtype)
    env = EnvelopeSpec(L.ENV_POLY, 0.0, L_BOX) if bc == "FBC" else NO_ENVELOPE
    Xg = torch.tensor(X, dtype=dtype, device="cuda")
    fg = None if g is None else torch.tensor(g, dtype=dtype, device="cuda")
    if isinstance(kappa, np.ndarray):
        spec, bg = ProgramSpec(L.PROG_RITZ_VALUE, alpha), torch.tensor(kappa, dtype=dtype, device="cuda")
    else:
        spec, bg = ProgramSpec(L.PROG_RITZ_VALUE, alpha, beta_const=kappa), None
    with pb.ops.kernel_path(path):
        loss = residual_means(_Holder(m, bc), Xg, spec, env, f=fg, beta=bg)[0]
        loss.backward()
        family = pb.ops.last_kernel_path()
        code = L.load().pde_last_kernel_path()
    assert code == (1 if family == "tcgen05" else 0)
    return float(loss.detach()), _grads(m), family


@pytest.mark.parametrize("bc", ["RB", "FBC"])
@pytest.mark.parametrize("act", ["sin", "tanh"])
@pytest.mark.parametrize("d", [1, 2, 3, 5])
def test_ritz_value_program_matches_oracle_on_both_families(d, act, bc):
    """The four (beta, f) combinations: constant / per-point beta, g given / NULL (constant alpha), at >= 4096 points.
    Generic kernel in float64 and float32, tensor-core kernel in float32."""
    rng = np.random.default_rng(300 + 100 * d + (act == "tanh") * 10 + (bc == "FBC"))
    net = _net(rng, d, 32, 4, act)
    for i in range(4):
        n = 4096 + 37 * i
        X = _f32(rng.uniform(0.0, L_BOX, (n, d)))
        g = _f32(rng.normal(size=n)) if i % 2 == 0 else None
        kappa = _f32(rng.uniform(0.5, 1.5, n)) if i // 2 == 0 else 0.75 * (i - 1)
        alpha = 0.37 if g is not None else (-1.0 if i == 1 else 0.6)     # (ignored when g is given)
        want, wgrads = _oracle(net, X, g, bc, alpha, kappa)
        got, ggrads, fam = _kernel(net, X, g, bc, alpha, kappa, torch.float64, "simt")
        assert fam == "simt_fma"
        assert abs(got - want) <= 1e-10 * max(abs(want), 1e-3), (i, got, want)
        e, where = grads_err(ggrads, wgrads)
        assert e <= 1e-10, (i, "simt f64", where, e)
        bar = max(1e-5, 2.0 * _e32(net, X, g, bc, alpha, kappa))
        for path, want_fam in (("simt", "simt_fma"), ("tc", "tcgen05")):
            got, ggrads, fam = _kernel(net, X, g, bc, alpha, kappa, torch.float32, path)
            assert fam == want_fam
            assert abs(got - want) <= bar * max(abs(want), 1e-3), (i, path, got, want, bar)
            e, where = grads_err(ggrads, wgrads)
            assert e <= bar, (i, path, where, e, bar)


def test_ritz_value_tensor_core_at_scale_matches_generic_fp64():
    rng = np.random.default_rng(2020)
    n, d = 1 << 20, 3
    net = _net(rng, d, 64, 4, "sin")
    X = _f32(rng.uniform(0.0, L_BOX, (n, d)))
    g = _f32(0.2 * rng.normal(size=n))
    kappa = _f32(rng.uniform(1.0, 2.0, n))
    want, wgrads, fam = _kernel(net, X, g, "RB", 0.0, kappa, torch.float64, "simt")
    assert fam == "simt_fma"
    got, ggrads, fam = _kernel(net, X, g, "RB", 0.0, kappa, torch.float32, "auto")
    assert fam == "tcgen05"
    assert abs(got - want) <= 1e-5 * abs(want), (got, want)
    e, where = grads_err(ggrads, wgrads)
    assert e <= 1e-5, (where, e)


# ---------------------------------------------------------------- drop-ins
def _torch_faces(per, d, mask, seed):
    """The torch.rand face draws of boundary_loss_dirichlet's face order, restricted to the mask (float64, cuda)."""
    torch.manual_seed(seed)
    blocks = []
    for i in range(d):
        for at_L in (False, True):
            if mask >> (2 * i + at_L) & 1:
                Xb = torch.rand(per, d, device="cuda", dtype=torch.float64) * L_BOX
                Xb[:, i] = L_BOX if at_L else 0.0
                blocks.append(Xb)
    return torch.cat(blocks).cpu()


@pytest.mark.parametrize("kappa", [0.0, 1.5])
@pytest.mark.parametrize("with_g", [True, False])
def test_boundary_energy_neumann_matches_oracle(with_g, kappa):
    import pde_b200 as pb
    d, per, mask = 3, 300, 0b011001
    torch.manual_seed(9)
    model = pb.poisson.SolutionNet(d, 32, 4, "RB").double().cuda()
    ref = copy.deepcopy(model).cpu()
    gfun = (lambda X: torch.sin(X).sum(dim=1)) if with_g else None
    torch.manual_seed(123)
    loss = pb.poisson.boundary_energy_neumann(model, L_BOX, per, d, "cuda", g=gfun, kappa=kappa, faces=mask)
    loss.backward()
    X = _torch_faces(per, d, mask, 123)
    want = boundary_energy(ref.net, X, mask, gfun(X) if with_g else None, L_BOX, "RB", kappa)
    if with_g or kappa:
        want.backward()
    assert abs(float(loss.detach()) - float(want.detach())) <= 1e-10 * abs(float(want.detach()))
    e, where = grads_err(_grads(model.net), _grads(ref.net))
    assert e <= 1e-10, (where, e)


def test_drm_plus_boundary_energy_is_the_ritz_functional():
    """drm_energy_loss + boundary_energy_neumann = E[u] / |Omega| of the specification on the same points, for a Robin
    condition on four faces of the box [0, 2]^3 (the other two keep the natural du/dn = 0)."""
    import pde_b200 as pb
    d, per, mask, kappa, ks = 3, 400, 0b110101, 0.8, [1, 2, 1]
    torch.manual_seed(4)
    model = pb.poisson.SolutionNet(d, 32, 4, "RB").double().cuda()
    ref = copy.deepcopy(model).cpu()
    X = torch.rand(3000, d, dtype=torch.float64) * L_BOX
    f = pb.poisson.rhs_f_for_u_sin(X, L_BOX, ks)
    gfun = lambda Z: torch.cos(Z).prod(dim=1)
    torch.manual_seed(77)
    Xc = X.cuda().requires_grad_(True)
    e = (pb.poisson.drm_energy_loss(model, Xc, f.cuda(), L_BOX)
         + pb.poisson.boundary_energy_neumann(model, L_BOX, per, d, "cuda", g=gfun, kappa=kappa, faces=mask))
    e.backward()
    Xb = _torch_faces(per, d, mask, 77)
    want = ritz_energy(ref.net, X.clone().requires_grad_(True), f, Xb, mask, gfun(Xb), L_BOX, "RB", kappa)
    want.backward()
    assert abs(float(e.detach()) - float(want.detach())) <= 1e-10 * abs(float(want.detach()))
    err, where = grads_err(_grads(model.net), _grads(ref.net))
    assert err <= 1e-10, (where, err)


@pytest.mark.parametrize("dtype,path", [(torch.float64, "simt"), (torch.float32, "tc")])
def test_mean_value_loss_matches_autograd(dtype, path):
    import pde_b200 as pb
    torch.manual_seed(6)
    model = pb.poisson.SolutionNet(2, 64, 4, "RB").double()
    with torch.no_grad():
        for p in model.parameters():
            p.copy_(p.float().double())      # weights the float32 kernel sees exactly
    ref = copy.deepcopy(model)
    m = copy.deepcopy(model).to("cuda", dtype)
    X = (torch.rand(5000, 2, dtype=torch.float64) * L_BOX).float().double()
    c = 0.3
    with pb.ops.kernel_path(path):
        loss = pb.poisson.mean_value_loss(m, X.to("cuda", dtype), L_BOX, c)
        loss.backward()
        assert pb.ops.last_kernel_path() == ("tcgen05" if path == "tc" else "simt_fma")
    want = mean_value_loss(ref.net, X, L_BOX, "RB", c)
    want.backward()
    bar = 1e-10 if dtype == torch.float64 else 1e-5
    assert abs(float(loss.detach()) - float(want.detach())) <= bar * max(abs(float(want.detach())), 1e-3)
    e, where = grads_err(_grads(m.net), _grads(ref.net))
    assert e <= bar, (where, e)


# ---------------------------------------------------------------- FusedTrainer against a reference-style loop
CASES = {
    # name: (method, form, faces, kappa, ks, extra trainer kwargs)
    "a_ritz_robin_all_faces": ("DRM", "ritz", 0b1111, 1.0, [1.0, 2.0], {}),
    "b_ritz_neumann_axis1_dirichlet_axis0": ("DRM", "ritz", 0b1100, 0.0, [1.0, 2.0], {"weights": {"pde": 1.0, "bc": 50.0}}),
    "c_ritz_pure_neumann_mean": ("DRM", "ritz", 0b1111, 0.0, [1.0, 2.0], {"mean_value": True, "weight_mean": 2.0}),
    "penalty_robin_noninteger_ks_mean": ("PINN", "penalty", 0b1111, 0.8, [0.75, 1.5],
                                         {"weight_neumann": 3.0, "mean_value": True}),
}


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("case", sorted(CASES))
def test_trainer_ritz_and_robin_match_reference_loop(case, graph):
    """RB model, d = 2.  Five epochs equal the reference-style loop (specification losses + torch.optim.Adam, float64 on
    the CPU) run on the trainer's own face points, with g = du*/dn + kappa u* from autograd of u*."""
    import pde_b200 as pb
    from oracle import autograd_ref as AR
    method, form, mask, kappa, ks, extra = CASES[case]
    torch.manual_seed(17)
    L, dim, n, epochs = L_BOX, 2, 1500, 5
    model = pb.poisson.SolutionNet(dim, 24, 4, "RB").double()
    ref = copy.deepcopy(model)
    model = model.cuda()
    X = torch.rand(n, dim, dtype=torch.float64) * L
    f = pb.poisson.rhs_f_for_u_sin(X, L, ks)
    tr = pb.train.FusedTrainer(model, L, ks, method=method, X=X.cuda(), f=f.cuda(), lr=2e-3, n_boundary=400,
                               neumann_faces=mask, neumann_form=form, robin_kappa=kappa, graph=graph, seed=5, **extra)
    w = tr.w
    nf = bin(mask).count("1")
    if form == "ritz":
        assert w["neumann"] == w["pde"] * nf / L
    want_rows = ["pde"] + (["bc"] if mask != 0b1111 else []) + ["neumann"] + (["mean"] if extra.get("mean_value") else [])
    assert tr.rows == want_rows and tr.nn == 100 * nf
    draws, terms = [], []
    for _ in range(epochs):
        tr.step(1)
        draws.append((tr.Xb.detach().cpu().clone() if tr.use["bc"] else None, tr.Xn.detach().cpu().clone(),
                      tr.gn.detach().cpu().clone()))
        terms.append({k: float(v) for k, v in tr.terms.items()})
    opt = torch.optim.Adam(ref.parameters(), lr=2e-3)
    c_star = exact_mean(L, ks)
    for ep in range(epochs):
        Xb, Xn, gn = draws[ep]
        g = _g_autograd(Xn, ks, mask) + kappa * pb.poisson.exact_u_prod_sin(Xn, L, ks).reshape(-1)
        assert float((gn - g).abs().max()) <= 1e-12
        opt.zero_grad()
        pde = (AR.pinn_loss if method == "PINN" else AR.drm_loss)(ref.net, X.clone().requires_grad_(True), f, L, "RB")
        parts = {"pde": (pde, w["pde"])}
        if Xb is not None:
            parts["bc"] = (torch.mean(ref(Xb, L) ** 2), w["bc"])
        if form == "ritz":
            parts["neumann"] = (ritz_value_loss(ref.net, Xn, g, L, "RB", kappa), w["pde"] * nf / L)
        else:
            parts["neumann"] = (flux_loss(ref.net, Xn.clone().requires_grad_(True), mask, g, L, "RB", kappa=kappa),
                                extra.get("weight_neumann", 1.0))
        if extra.get("mean_value"):
            parts["mean"] = (mean_value_loss(ref.net, X, L, "RB", c_star), extra.get("weight_mean", 1.0))
        total = sum(v * wt for v, wt in parts.values())
        for nm, want in [(k, float(v.detach())) for k, (v, _) in parts.items()] + [("total", float(total.detach()))]:
            assert abs(terms[ep][nm] - want) <= 1e-9 * max(1.0, abs(want)), (ep, nm, terms[ep][nm], want)
        total.backward()
        opt.step()
    for a, b in zip(model.parameters(), ref.parameters()):
        assert float((a.detach().cpu() - b.detach()).abs().max()) <= 1e-9 * max(1.0, float(b.detach().abs().max()))
    assert not torch.equal(draws[0][1], draws[1][1])


def _launches_per_epoch(tr):
    import pde_b200 as pb
    tr.step(1)
    torch.cuda.synchronize()
    before = pb.ops.launch_count()
    tr.step(1)
    return pb.ops.launch_count() - before


def test_trainer_defaults_keep_rows_and_launches():
    """Without the new arguments the Neumann row is the penalty of weight 1 and there is no 'mean' row.  Robin data
    costs one library launch per epoch (u* on the face points); the mean constraint costs two residual calls (sums, then
    the seeded reverse sweep) of three launches each (parameter pack, fused kernel, reduction); the Ritz form costs
    nothing over the penalty."""
    import pde_b200 as pb
    mk = lambda **kw: pb.train.FusedTrainer(pb.poisson.SolutionNet(2, 16, 3, "RB").cuda(), 2.0, [1, 1], n_interior=512,
                                            neumann_faces=0b0011, graph=False, **kw)
    tr = mk()
    assert tr.rows == ["pde", "bc", "neumann"] and tr.w["neumann"] == 1.0 and "mean" not in tr.w
    assert tr.nspec.kind == 5 and tr.nspec.beta_const == 0.0
    base = _launches_per_epoch(tr)
    assert "mean" not in tr.terms
    assert _launches_per_epoch(mk(robin_kappa=0.5)) == base + 1
    assert _launches_per_epoch(mk(mean_value=True)) == base + 6
    assert _launches_per_epoch(mk(method="DRM", neumann_form="ritz")) == base


# ---------------------------------------------------------------- convergence (tools/ritz_convergence.py, case (a))
# The recorded run (profiles/ritz_convergence.json, NVIDIA B200 at a 1000 W power limit) reached a best L2 error of
# 5.85e-3 in case (a), Ritz form, within 4000 epochs; the bound leaves a margin of 2.5x.
CONV_EPOCHS = 4000
CONV_BOUND = 0.015


def test_ritz_robin_case_a_converges():
    """Case (a) of tools/ritz_convergence.py (Robin, kappa = 1, on every face; DRM with the Ritz boundary term), same
    seeds as the recorded run."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "tools"))
    import ritz_convergence as RC
    _, rec = RC.run_case("a", "ritz", CONV_EPOCHS, seed=0)
    assert rec["best_l2"] <= CONV_BOUND, rec["best_l2"]


# ---------------------------------------------------------------- two or more GPUs (harness as in test_gpu_multi.py)
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _entry(rank, world, port):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        _w_exchange(rank, world)
    finally:
        dist.barrier()
        dist.destroy_process_group()


def _w_exchange(rank, world):
    """The Ritz value program with group= and the exchange folded into the NVLink reduction equals the single big batch,
    for the boundary energy form (per-point beta and g) and for the mean constraint."""
    import torch.distributed as dist
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import NO_ENVELOPE, ProgramSpec, residual_mean
    n_loc = 6000
    torch.manual_seed(3)
    m = pb.poisson.SolutionNet(3, 64, 5, "RB").cuda()
    X = torch.rand(n_loc * world, 3, device="cuda") * L_BOX
    g = torch.cos(X).sum(dim=1)
    beta = 1.0 + X[:, 0]
    spec = ProgramSpec(L.PROG_RITZ_VALUE, 0.0)
    sl = slice(rank * n_loc, (rank + 1) * n_loc)
    pb.ops.use_nvlink_exchange(None, 1 << 15, torch.float32)
    for fn in (lambda Z, s, grp: residual_mean(m, Z, spec, NO_ENVELOPE, f=g[s], beta=beta[s], group=grp),
               lambda Z, s, grp: pb.poisson.mean_value_loss(m, Z, L_BOX, 0.1, group=grp)):
        m.zero_grad()
        big = fn(X, slice(None), None)
        big.backward()
        want = [p.grad.clone() for p in m.parameters()]
        m.zero_grad()
        part = fn(X[sl], sl, dist.group.WORLD)
        part.backward()
        assert pb.ops.last_kernel_path() == "tcgen05"
        assert abs(float(part) - float(big)) <= 2e-6 * max(abs(float(big)), 1e-3), (float(part), float(big))
        for p, w in zip(m.parameters(), want):
            assert float((p.grad - w).abs().max()) <= 1e-5 * float(w.abs().max())
    pb.ops._EXCHANGE[(dist.group.WORLD, torch.float32)].check()


def test_ritz_value_folded_exchange_matches_single_batch():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_entry, args=(2, _free_port()), nprocs=2, join=True)
