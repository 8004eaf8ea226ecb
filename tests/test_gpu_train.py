"""GPU tests of the epoch pieces around the loss step (pde_b200.train; SURVEY.md §8f-1, §8f-3):
point sampling + manufactured right-hand side, fused Adam, the CUDA-graph epoch against the
reference's loop (its nested-autograd loss + torch.optim.Adam, run on the CPU in float64 through
oracle/autograd_ref.py), and device-side best-model tracking."""
import math

import numpy as np
import pytest
import torch

import pde_b200 as pb
from oracle import autograd_ref as AR

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("dim", [1, 3, 5])
def test_sampling_and_rhs(dim, dtype):
    L, ks, n = 2.0, [1 + (i % 3) for i in range(dim)], 1 << 18
    X, u, f = pb.train.sample_points_rhs(n, dim, L, ks, dtype=dtype, seed=7, offset=3, want_u=True)
    assert X.shape == (n, dim) and X.dtype == dtype
    assert float(X.min()) >= 0.0 and float(X.max()) < L          # half-open like torch.rand * L
    Xd = X.double()
    assert abs(float(Xd.mean()) - L / 2) < 4 * (L / math.sqrt(12)) / math.sqrt(n * dim) * 1.5
    assert abs(float(Xd.var()) - L * L / 12) < 0.01
    # coordinates are independent of each other and of the neighbouring point
    if dim > 1:
        c = torch.corrcoef(Xd.T)
        assert float((c - torch.eye(dim, device=c.device, dtype=c.dtype)).abs().max()) < 0.01
    assert abs(float(torch.corrcoef(torch.stack([Xd[:-1, 0], Xd[1:, 0]]))[0, 1])) < 0.01
    # manufactured solution / rhs against the reference formulas (Poisson_ND.py:49-58)
    tol = 1e-12 if dtype == torch.float64 else 2e-6
    uw, fw = pb.poisson.exact_u_prod_sin(X, L, ks), pb.poisson.rhs_f_for_u_sin(X, L, ks)
    assert float((u - uw).abs().max()) <= tol
    assert float((f - fw).abs().max()) <= tol * float(fw.abs().max())
    # counter-based: same (seed, offset) -> same points; another offset or seed -> other points
    X2, _, _ = pb.train.sample_points_rhs(n, dim, L, ks, dtype=dtype, seed=7, offset=3)
    assert torch.equal(X, X2)
    X3, _, _ = pb.train.sample_points_rhs(n, dim, L, ks, dtype=dtype, seed=7, offset=4)
    X4, _, _ = pb.train.sample_points_rhs(n, dim, L, ks, dtype=dtype, seed=8, offset=3)
    assert not torch.equal(X, X3) and not torch.equal(X, X4)
    # evaluation at given points
    _, u5, f5 = pb.train.sample_points_rhs(0, 0, L, ks, X=X, want_u=True)
    assert torch.equal(u5, u) and torch.equal(f5, f)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_fused_adam_matches_torch_adam(dtype):
    torch.manual_seed(0)
    shapes = [(16, 3), (16,), (16, 16), (16,), (1, 16), (1,), ()]     # last: a trainable energy scalar
    ours = [torch.randn(s, dtype=dtype, device="cuda") for s in shapes]
    theirs = [p.clone().requires_grad_(True) for p in ours]
    opt_t = torch.optim.Adam(theirs, lr=1e-3)
    opt = pb.train.FusedAdam(ours, lr=1e-3)
    n = sum(p.numel() for p in ours)
    for it in range(12):
        g = torch.randn(n + 3, dtype=dtype, device="cuda") * (10.0 ** (it % 3 - 1))
        o = 0
        for p in theirs:
            p.grad = (0.5 * g[o:o + p.numel()]).view_as(p).clone(); o += p.numel()
        opt_t.step()
        opt.step(g, grad_scale=0.5)
    assert int(opt.step_count) == 12
    tol = 1e-12 if dtype == torch.float64 else 2e-6
    for a, b in zip(ours, theirs):
        assert float((a - b.detach()).abs().max()) <= tol * max(1.0, float(b.detach().abs().max()))


def _reference_loop(model64_cpu, X, f, L, bc, method, lr, epochs):
    """train_poisson_nd's PINN / DRM branch (Poisson_ND.py:215-241) restated with the oracle's
    nested-autograd loss: loss -> backward -> torch.optim.Adam.step(), float64 on the CPU."""
    net = model64_cpu.net
    opt = torch.optim.Adam(net.parameters(), lr=lr)
    losses = []
    for _ in range(epochs):
        loss, gflat = AR.loss_and_grads(method, net, X, f, L, bc)
        o = 0
        for p in net.parameters():
            p.grad = gflat[o:o + p.numel()].view_as(p).clone(); o += p.numel()
        opt.step()
        losses.append(loss)
    return losses


@pytest.mark.parametrize("method,bc,dim", [("PINN", "FBC", 2), ("DRM", "RB", 3), ("PINN", "FBC", 3)])
@pytest.mark.parametrize("graph", [True, False])
def test_trainer_matches_reference_loop(method, bc, dim, graph):
    torch.manual_seed(11)
    L, ks, N, lr, epochs = 2.0, [1] * dim, 4096 + 37, 1e-3, 6
    m_cpu = pb.poisson.SolutionNet(dim, 32, 4, bc).double()
    m_gpu = pb.poisson.SolutionNet(dim, 32, 4, bc).double()
    m_gpu.load_state_dict(m_cpu.state_dict())
    m_gpu = m_gpu.cuda()
    X = torch.rand(N, dim, dtype=torch.float64) * L
    f = pb.poisson.rhs_f_for_u_sin(X, L, ks)
    want = _reference_loop(m_cpu, X, f, L, bc, method.lower(), lr, epochs)
    # PDE term only: an 'RB' model with weights={'bc': 0} is the raw network without boundary term (the natural-BC
    # reading of BASELINE config 3); the reference's own default for 'RB' is bc = 1e4 (covered further down)
    tr = pb.train.FusedTrainer(m_gpu, L, ks, method=method, lr=lr, X=X.cuda(), f=f.cuda(), history=epochs, graph=graph,
                               weights={"bc": 0.0})
    tr.step(epochs)
    got = tr.hist_loss.cpu().numpy()
    np.testing.assert_allclose(got, np.array(want), rtol=1e-9, atol=1e-12)
    for a, b in zip(m_gpu.parameters(), m_cpu.parameters()):
        assert float((a.detach().cpu() - b.detach()).abs().max()) <= 1e-9 * max(1.0, float(b.detach().abs().max()))
    assert int(tr.opt.step_count) == epochs and tr.epochs_done == epochs


def test_trainer_fp32_tensor_core_path_and_best_tracking():
    """Config-2 shaped network on the tcgen05 path: graph replays are deterministic, the L2 history's minimum
    is what keep_best kept, and load_best restores those parameters."""
    torch.manual_seed(5)
    L, ks = 2.0, [1, 1, 1]
    def run():
        torch.manual_seed(5)
        m = pb.poisson.SolutionNet(3, 64, 5, "FBC").cuda()
        tr = pb.train.FusedTrainer(m, L, ks, method="PINN", n_interior=1 << 14, lr=2e-3, n_test=4096, history=20, seed=3)
        tr.step(20)
        return m, tr
    m1, t1 = run()
    m2, t2 = run()
    for a, b in zip(m1.parameters(), m2.parameters()):
        assert torch.equal(a, b)
    h = t1.hist_l2sq.double().cpu().numpy()
    assert h.min() > 0 and abs(float(t1.best_metric) / 4096 - h.min()) <= 1e-6 * h.min()
    assert int(t1.best_step) == int(np.argmin(h)) + 1
    assert abs(float(t1.l2) - math.sqrt(h[-1])) <= 1e-6
    losses = t1.hist_loss.cpu().numpy()
    assert losses[-1] < losses[0]                      # Adam makes progress on the PINN residual
    # the kept parameters reproduce the best metric on the same test draw
    t1.load_best()
    Xt, ut, _ = pb.train.sample_points_rhs(4096, 3, L, ks, seed=3 ^ 0x9E3779B97F4A7C15, offset=int(t1.best_step), want_u=True)
    with torch.no_grad():
        l2sq = float(((m1(Xt, L) - ut) ** 2).mean())
    assert abs(l2sq - h.min()) <= 2e-5 * h.min()


def test_trainer_resamples_every_epoch():
    torch.manual_seed(1)
    m = pb.poisson.SolutionNet(2, 32, 4, "FBC").cuda()
    tr = pb.train.FusedTrainer(m, 2.0, [1, 2], method="DRM", n_interior=8192, resample=True, seed=9, history=4)
    seen = []
    for _ in range(4):
        tr.step()
        seen.append(tr.X.clone())
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[2], seen[3])
    # epoch e draws the points of Philox offset e (the step counter before the update)
    for e in (0, 1, 3):
        Xe, _, fe = pb.train.sample_points_rhs(8192, 2, 2.0, [1, 2], seed=9, offset=e)
        assert torch.equal(seen[e], Xe)
    assert torch.isfinite(tr.hist_loss).all()


def test_wan_frozen_jets_give_identical_losses_and_grads():
    """§8f-2: the critic steps reuse the frozen u-network's jets on fixed points (IPW_1D_WAN.py:186-194)."""
    from pde_b200.schrodinger import ipw_1d_wan as W
    torch.manual_seed(2)
    L, n = 2.0, 2
    um = W.FCN([1, 50, 50, 50, 1], L=L, enforce_bc=True).cuda()
    vm = W.FCN([1, 20, 20, 20, 1], L=L).cuda()
    x = torch.linspace(0, L, 1000, device="cuda").view(-1, 1).requires_grad_(True)
    for p in um.parameters():
        p.requires_grad_(False)
    _, lv_a, lp_a, _ = W.WAN_loss(um, vm, x, n, L)
    lv_a.backward()
    ga = [p.grad.clone() for p in vm.parameters()]
    for p in vm.parameters():
        p.grad = None
    Ju = pb.frozen_jets(um, x)
    _, lv_b, lp_b, _ = W.WAN_loss(um, vm, x, n, L, u_jets=Ju)
    lv_b.backward()
    assert torch.equal(lv_a, lv_b) and torch.equal(lp_a, lp_b)
    for a, p in zip(ga, vm.parameters()):
        assert torch.equal(a, p.grad)
    assert all(p.grad is None for p in um.parameters())
    with pytest.raises(ValueError):
        W.WAN_loss(um, vm, x, n, L, u_jets=Ju[:10])


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("set_to_none", [False, True])
def test_train_adam_dropin_matches_torch_adam(graph, set_to_none):
    """pb.train.Adam (one flat gradient vector, one pde_adam_step launch per step) follows torch.optim.Adam through a
    reference-style epoch on the QHO 2-D PINN loss, eagerly and as a replayed CUDA graph — with the gradients adopted
    from the loss operator's own buffer (zero_grad(): no fill, no per-parameter accumulation) and with the optimiser's
    own views (set_to_none=False)."""
    from pde_b200.schrodinger import qho_2d as Q
    g1 = torch.linspace(-6.0, 6.0, 40, dtype=torch.float64)
    xg, yg = torch.meshgrid(g1, g1, indexing="ij")
    xd, yd = xg.cuda(), yg.cuda()
    E = Q.Exact_energy(2, 1, 6.0)

    def build(kind):
        torch.manual_seed(11)
        m = Q.FCN([2, 24, 24, 24, 1], 2, 1, "FBC").double().cuda()
        opt = (pb.train.Adam(m.parameters(), lr=2e-3, weight_decay=1e-4) if kind == "fused"
               else torch.optim.Adam(m.parameters(), lr=2e-3, weight_decay=1e-4))   # (capturable=True keeps its step count, hence
                                                                                      #  the bias corrections, in float32: 6e-6 off per step)

        def epoch():
            opt.zero_grad(set_to_none=set_to_none)
            l = Q.PINN_loss(m, xd, yd, E, 6.0)
            l.backward()
            opt.step()
            return l.detach()
        return m, epoch, opt
    m_ref, ep_ref, _ = build("torch")
    for _ in range(7):
        l_ref = ep_ref()
    m_new, ep_new, opt_new = build("fused")
    if graph:
        ge = pb.train.GraphedEpoch(ep_new, warmup=3)
        ge()                       # 3 eager epochs + capture
        for _ in range(4):
            l_new = ge()           # 4 replays
    else:
        for _ in range(7):
            l_new = ep_new()
    torch.cuda.synchronize()
    assert abs(float(l_new) - float(l_ref)) <= 1e-9 * abs(float(l_ref))
    for a, b in zip(m_new.parameters(), m_ref.parameters()):
        assert float((a - b).abs().max()) <= 1e-9 * max(1.0, float(b.abs().max()))
    # every step read the gradients where they were (the operator's buffer or the optimiser's own): nothing gathered
    assert opt_new.gathered_steps == 0 and opt_new.adopted_steps == (4 if graph else 7)


def test_graphed_wan_epoch_matches_eager():
    """One epoch of the IPW 1-D WAN loop (5 critic steps + 1 solution step, IPW_1D_WAN.py:186-208) captured as a
    CUDA graph equals the same epoch run eagerly."""
    from pde_b200.schrodinger import ipw_1d_wan as W
    L, n = 2.0, 2
    x = torch.linspace(0, L, 1000, device="cuda").view(-1, 1)

    def build():
        torch.manual_seed(4)
        um = W.FCN([1, 50, 50, 50, 1], L=L, enforce_bc=True).cuda()
        vm = W.FCN([1, 20, 20, 20, 1], L=L).cuda()
        ou = torch.optim.Adam(um.parameters(), lr=1e-3, capturable=True)
        ov = torch.optim.Adam(vm.parameters(), lr=1e-3, capturable=True)

        def epoch():
            Ju = pb.frozen_jets(um, x)
            for _ in range(5):
                ov.zero_grad(set_to_none=False)
                _, lv, _, _ = W.WAN_loss(um, vm, x, n, L, u_jets=Ju)
                gv = torch.autograd.grad(lv, list(vm.parameters()))
                for p, g in zip(vm.parameters(), gv):
                    p.grad = g if p.grad is None else p.grad.copy_(g)
                ov.step()
            ou.zero_grad(set_to_none=False)
            total, _, lp, ln = W.WAN_loss(um, vm, x, n, L)
            gu = torch.autograd.grad(total, list(um.parameters()))
            for p, g in zip(um.parameters(), gu):
                p.grad = g if p.grad is None else p.grad.copy_(g)
            ou.step()
            return total.detach()
        return um, vm, epoch

    um1, vm1, ep1 = build()
    for _ in range(6):
        t1 = ep1()
    um2, vm2, ep2 = build()
    g = pb.train.GraphedEpoch(ep2, warmup=3)
    g()                      # 3 eager epochs + capture
    for _ in range(3):
        t2 = g()             # 3 replays
    torch.cuda.synchronize()
    assert g.replays == 3
    for a, b in zip(list(um1.parameters()) + list(vm1.parameters()), list(um2.parameters()) + list(vm2.parameters())):
        assert float((a - b).abs().max()) <= 1e-6 * max(1.0, float(a.abs().max()))
    assert abs(float(t1) - float(t2)) <= 1e-5 * max(1e-3, abs(float(t1)))


# ---------------------------------------------------------------- the rest of the reference epoch (Poisson_ND.py:224-276)
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("method,norm_mode", [("PINN", "nontrivial"), ("DRM", "l2")])
def test_trainer_rb_bc_data_norm_terms_match_reference_loop(method, norm_mode, graph):
    """RB branch with the soft Dirichlet penalty on freshly drawn face points, the data term and the norm term
    (Poisson_ND.py:224-239): five epochs of the fused trainer equal the reference loop (oracle nested-autograd losses +
    torch.optim.Adam, float64 on the CPU) run on the face points the trainer drew."""
    import copy
    torch.manual_seed(11)
    L, ks, dim, n, nd, epochs = 2.0, [1, 2], 2, 1500, 120, 5
    w = {"pde": 1.0, "bc": 50.0, "data": 20.0, "norm": 0.3}
    model = pb.poisson.SolutionNet(dim, 24, 4, "RB").double()
    ref = copy.deepcopy(model)
    model = model.cuda()
    X = torch.rand(n, dim, dtype=torch.float64) * L
    f = pb.poisson.rhs_f_for_u_sin(X, L, ks)
    Xd = torch.rand(nd, dim, dtype=torch.float64) * L
    ud = pb.poisson.exact_u_prod_sin(Xd, L, ks)
    tr = pb.train.FusedTrainer(model, L, ks, method=method, X=X.cuda(), f=f.cuda(), lr=2e-3, weights=w, n_boundary=400,
                               X_data=Xd.cuda(), u_data=ud.cuda(), norm_mode=norm_mode, graph=graph, seed=5)
    faces, terms = [], []
    for _ in range(epochs):
        tr.step(1)
        faces.append(tr.Xb.detach().cpu().clone())
        terms.append({k: float(v) for k, v in tr.terms.items()})
    # reference loop on the same face points
    opt = torch.optim.Adam(ref.parameters(), lr=2e-3)
    for ep in range(epochs):
        opt.zero_grad()
        Xr = X.clone().requires_grad_(True)
        pde = (AR.pinn_loss if method == "PINN" else AR.drm_loss)(ref.net, Xr, f, L, "RB")
        bc = torch.mean(ref(faces[ep], L) ** 2)                 # equal face counts: mean of face means = overall mean
        data = torch.mean((ref(Xd, L) - ud) ** 2)
        nrm = pb.poisson.norm_loss(ref(X, L), mode=norm_mode)
        total = w["pde"] * pde + w["bc"] * bc + w["data"] * data + w["norm"] * nrm
        for got, want, nm in ((terms[ep]["pde"], pde, "pde"), (terms[ep]["bc"], bc, "bc"), (terms[ep]["data"], data, "data"),
                              (terms[ep]["norm"], nrm, "norm"), (terms[ep]["total"], total, "total")):
            assert abs(got - float(want)) <= 1e-9 * max(1.0, abs(float(want))), (ep, nm, got, float(want))
        total.backward(); opt.step()
    for a, b in zip(model.parameters(), ref.parameters()):
        assert float((a.detach().cpu() - b.detach()).abs().max()) <= 1e-9 * max(1.0, float(b.detach().abs().max()))
    # the face draw: 2d faces with equal counts, the face coordinate exactly 0 or L, the others inside [0, L)
    Xb = faces[-1].view(2 * dim, -1, dim)
    for k in range(2 * dim):
        assert torch.all(Xb[k, :, k // 2] == (L if k % 2 else 0.0))
    assert float(faces[-1].min()) >= 0.0 and float(faces[-1].max()) <= L and not torch.equal(faces[0], faces[1])
    with pytest.raises(ValueError):
        pb.train.FusedTrainer(model, L, ks, weights={"bogus": 1.0})
    with pytest.raises(ValueError):
        pb.train.WanTrainer(model, pb.poisson.CriticNet(dim, 8, 2).double().cuda(), L, ks, weights={"bogus": 1.0})
    with pytest.raises(ValueError):
        pb.train.FusedTrainer(model, L, ks, weights={"data": 1.0})      # data weight without data points


def test_trainer_default_weights_follow_reference():
    """weights default like Poisson_ND.py:169-173: bc 1e4 for an 'RB' model (soft constraint), 0 for 'FBC'."""
    m = pb.poisson.SolutionNet(2, 16, 3, "RB").cuda()
    tr = pb.train.FusedTrainer(m, 2.0, [1, 1], n_interior=512, graph=False)
    assert tr.w["bc"] == 1e4 and tr.use["bc"] and tr.w["data"] == 0.0 and not tr.use["norm"]
    tr.step(2)
    assert float(tr.terms["bc"]) > 0.0 and math.isfinite(float(tr.terms["total"]))
    m2 = pb.poisson.SolutionNet(2, 16, 3, "FBC").cuda()
    tr2 = pb.train.FusedTrainer(m2, 2.0, [1, 1], n_interior=512, graph=False)
    assert tr2.w["bc"] == 0.0 and tr2.rows == ["pde"]


def test_wan_trainer_matches_reference_loop():
    """The WAN branch of the reference epoch (Poisson_ND.py:242-276: critic_steps critic updates and one solution
    update per epoch, every evaluation on freshly drawn points): four epochs of WanTrainer (drop-in wan_losses on the
    fused kernels + torch Adam) equal the reference loop (oracle nested-autograd wan_losses + torch.optim.Adam, float64
    on the CPU) run on the points the trainer drew."""
    import copy
    torch.manual_seed(13)
    L, ks, dim, n, epochs, csteps, reg = 2.0, [1, 1], 2, 800, 4, 3, 0.7
    w = {"pde": 1.0, "bc": 30.0, "data": 5.0, "norm": 0.2}
    um = pb.poisson.SolutionNet(dim, 24, 4, "RB").double()
    vm = pb.poisson.CriticNet(dim, 16, 3).double()
    ur, vr = copy.deepcopy(um), copy.deepcopy(vm)
    um, vm = um.cuda(), vm.cuda()
    Xd = torch.rand(60, dim, dtype=torch.float64) * L
    ud = pb.poisson.exact_u_prod_sin(Xd, L, ks)
    tr = pb.train.WanTrainer(um, vm, L, ks, n_interior=n, lr=2e-3, critic_steps=csteps, wan_reg=reg, weights=w, n_boundary=200,
                             X_data=Xd.cuda(), u_data=ud.cuda(), norm_mode="l2", seed=3, graph=False, record_points=True)
    hist = []
    for _ in range(epochs):
        tr.step(1)
        hist.append({k: float(v) for k, v in tr.last.items()})
    draws = iter(tr.drawn)
    opt_u = torch.optim.Adam(ur.parameters(), lr=2e-3)
    opt_v = torch.optim.Adam(vr.parameters(), lr=2e-3)
    for ep in range(epochs):
        for _ in range(csteps):
            kind, Xc, fc = next(draws); assert kind == "v"
            Xc = Xc.cpu().requires_grad_(True)
            _, lv, _, _ = AR.wan_losses(ur.net, vr.net, Xc, fc.cpu(), L, "RB", v_reg_weight=reg)
            opt_v.zero_grad(); lv.backward(); opt_v.step()
        kind, Xu, fu = next(draws); assert kind == "u"
        Xu = Xu.cpu().requires_grad_(True)
        lpde, _, weak, pn = AR.wan_losses(ur.net, vr.net, Xu, fu.cpu(), L, "RB", v_reg_weight=reg)
        kind, Xb, _ = next(draws); assert kind == "bc"
        bc = torch.mean(ur(Xb.cpu(), L) ** 2)
        data = torch.mean((ur(Xd, L) - ud) ** 2)
        nrm = pb.poisson.norm_loss(ur(Xu.detach(), L), mode="l2")
        total = w["pde"] * lpde + w["bc"] * bc + w["data"] * data + w["norm"] * nrm
        for nm, want in (("pde", lpde), ("bc", bc), ("data", data), ("norm", nrm), ("total", total), ("wan_loss_v", lv),
                         ("wan_weak", weak), ("wan_phi_norm", pn)):
            assert abs(hist[ep][nm] - float(want)) <= 1e-9 * max(1.0, abs(float(want))), (ep, nm, hist[ep][nm], float(want))
        opt_u.zero_grad(); total.backward(); opt_u.step()
    for a, b in zip(list(um.parameters()) + list(vm.parameters()), list(ur.parameters()) + list(vr.parameters())):
        assert float((a.detach().cpu() - b.detach()).abs().max()) <= 1e-9 * max(1.0, float(b.detach().abs().max()))


def test_wan_trainer_graph_replays_draw_fresh_points():
    """Captured WAN epoch: every replay draws new points (device draw counter) and keeps training."""
    torch.manual_seed(2)
    um = pb.poisson.SolutionNet(2, 16, 3, "FBC").cuda()
    vm = pb.poisson.CriticNet(2, 16, 3).cuda()
    tr = pb.train.WanTrainer(um, vm, 2.0, [1, 1], n_interior=2048, critic_steps=2, graph=True)
    tr.step(1)
    X1 = tr.bufs[-1][0].detach().clone(); d1 = int(tr.draws)
    tr.step(3)
    assert int(tr.draws) == d1 + 3 * 3 and not torch.equal(X1, tr.bufs[-1][0].detach())
    assert all(math.isfinite(float(v)) for v in tr.last.values())
