"""GPU tests of Neumann / Robin boundary conditions: the boundary-flux program (PDE_PROG_FLUX) on both kernel families
against the float64 autograd specification (tests/flux_oracle.py), its refusals, the one-launch face sampler
(pde_sample_faces_rhs), the Poisson drop-in boundary_loss_neumann and the Neumann term of FusedTrainer.

Bars (DESIGN.md §7): float64 on the generic kernel 1e-10; float32 max(1e-5, 2 e32), e32 being the distance between the
specification run in float32 and in float64 on the same inputs (and on inputs one float32 ulp away)."""
import copy
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest
import torch

from conftest import grads_err
from flux_oracle import flux_loss, manufactured_flux

pytestmark = pytest.mark.gpu
L_BOX = 2.0


def _masks(d):
    """one face, both faces of one axis, every face, and a non-contiguous set"""
    out = [1 << (2 * d - 1), 3 << (2 * (d // 2)), (1 << 2 * d) - 1]
    if d == 2:
        out.append(0b1001)
    if d >= 3:
        out.append(0b100101)
    return out


def _face_points(rng, d, mask, per):
    ks = [k for k in range(2 * d) if mask >> k & 1]
    X = rng.uniform(0.0, L_BOX, (per * len(ks), d))
    for j, k in enumerate(ks):
        X[j * per:(j + 1) * per, k // 2] = L_BOX if k % 2 else 0.0
    return _f32(X)


def _f32(a):
    """values the float32 kernels see exactly"""
    return a.astype(np.float32).astype(np.float64)


def _net(rng, d, width, depth, act):
    """A reference-style SolutionNet-shaped Sequential (float64 master copy) with float32-representable weights."""
    import pde_b200 as pb
    mods, w_in = [], d
    for _ in range(depth - 1):
        mods += [torch.nn.Linear(w_in, width), pb.poisson.Sin() if act == "sin" else torch.nn.Tanh()]
        w_in = width
    mods += [torch.nn.Linear(w_in, 1)]
    net = torch.nn.Sequential(*mods).double()
    with torch.no_grad():
        for m in net:
            if isinstance(m, torch.nn.Linear):
                m.weight.copy_(torch.tensor(rng.uniform(-1, 1, m.weight.shape) / math.sqrt(m.weight.shape[1])).float().double())
                m.bias.copy_(torch.tensor(rng.uniform(-0.5, 0.5, m.bias.shape)).float().double())
    return net


class _Holder(torch.nn.Module):
    """``.net`` + ``.bc_mode``, so that the ops see the envelope the oracle applies."""

    def __init__(self, net, bc):
        super().__init__()
        self.net, self.bc_mode = net, bc


def _g(p):
    """p.grad as float64 numpy; autograd leaves it None for a parameter the loss does not reach (with kappa = 0 the
    output bias: it does not change grad u), where the kernels write zeros."""
    return np.zeros(tuple(p.shape)) if p.grad is None else p.grad.double().cpu().numpy()


def _grads(net):
    lin = [m for m in net if isinstance(m, torch.nn.Linear)]
    return [_g(m.weight) for m in lin], [_g(m.bias) for m in lin]


def _oracle(net, X, mask, g, bc, alpha, kappa, dtype=torch.float64):
    """(loss, grads) of the specification on the CPU in ``dtype``."""
    ref = copy.deepcopy(net).to(dtype)
    Xt = torch.tensor(X, dtype=dtype).requires_grad_(True)
    gt = None if g is None else torch.tensor(g, dtype=dtype)
    kt = torch.tensor(kappa, dtype=dtype) if isinstance(kappa, np.ndarray) else kappa
    loss = flux_loss(ref, Xt, mask, gt, L_BOX, bc, alpha=alpha, kappa=kt)
    loss.backward()
    return float(loss.detach()), _grads(ref)


def _e32(net, X, mask, g, bc, alpha, kappa, draws=8):
    """The specification's own float32 error (loss and gradients): the worst case over these inputs and eight inputs one
    float32 ulp away, as for the golden fixtures' e32_* figures (tests/conftest.py), because a single draw of a
    cancelling quantity is not representative."""
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
        l32, g32 = _oracle(netj, Xj, mask, gj, bc, alpha, kj, torch.float32)
        l64, g64 = _oracle(netj, Xj, mask, gj, bc, alpha, kj, torch.float64)
        worst = max(worst, abs(l32 - l64) / max(abs(l64), 1e-3), grads_err(g32, g64)[0])
    return worst


def _kernel(net, X, mask, g, bc, alpha, kappa, dtype, path):
    """loss and gradients of the FLUX program through ops.residual_means on the given kernel family."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import EnvelopeSpec, ProgramSpec, NO_ENVELOPE, residual_means
    m = copy.deepcopy(net).to("cuda", dtype)
    env = EnvelopeSpec(L.ENV_POLY, 0.0, L_BOX) if bc == "FBC" else NO_ENVELOPE
    Xg = torch.tensor(X, dtype=dtype, device="cuda")
    fg = None if g is None else torch.tensor(g, dtype=dtype, device="cuda")
    if isinstance(kappa, np.ndarray):
        spec, bg = ProgramSpec(L.PROG_FLUX, alpha, faces=mask), torch.tensor(kappa, dtype=dtype, device="cuda")
    else:
        spec, bg = ProgramSpec(L.PROG_FLUX, alpha, beta_const=kappa, faces=mask), None
    with pb.ops.kernel_path(path):
        loss = residual_means(_Holder(m, bc), Xg, spec, env, f=fg, beta=bg)[0]
        loss.backward()
        family = pb.ops.last_kernel_path()
    return float(loss.detach()), _grads(m), family


@pytest.mark.parametrize("bc", ["RB", "FBC"])
@pytest.mark.parametrize("act", ["sin", "tanh"])
@pytest.mark.parametrize("d", [1, 2, 3, 5])
def test_flux_program_matches_oracle_on_both_families(d, act, bc):
    """Every mask shape; the four (beta, f) combinations rotate over the masks (constant / per-point beta, g given /
    NULL).  Generic kernel in float64 and float32, tensor-core kernel in float32."""
    rng = np.random.default_rng(100 * d + (act == "tanh") * 10 + (bc == "FBC"))
    net = _net(rng, d, 32, 4, act)
    for i, mask in enumerate(_masks(d)):
        X = _face_points(rng, d, mask, 61 + 17 * i)
        n = X.shape[0]
        g = _f32(rng.normal(size=n)) if i % 2 == 0 else None
        kappa = _f32(rng.uniform(0.5, 1.5, n)) if (i // 2) % 2 == 0 else 0.25 * (i + 1)
        alpha = -1.3 if i == 1 else 1.0
        want, wgrads = _oracle(net, X, mask, g, bc, alpha, kappa)
        got, ggrads, fam = _kernel(net, X, mask, g, bc, alpha, kappa, torch.float64, "simt")
        assert fam == "simt_fma"
        assert abs(got - want) <= 1e-10 * max(abs(want), 1e-3), (mask, got, want)
        e, where = grads_err(ggrads, wgrads)
        assert e <= 1e-10, (mask, "simt f64", where, e)
        bar = max(1e-5, 2.0 * _e32(net, X, mask, g, bc, alpha, kappa))
        for path, want_fam in (("simt", "simt_fma"), ("tc", "tcgen05")):
            got, ggrads, fam = _kernel(net, X, mask, g, bc, alpha, kappa, torch.float32, path)
            assert fam == want_fam
            assert abs(got - want) <= bar * max(abs(want), 1e-3), (mask, path, got, want, bar)
            e, where = grads_err(ggrads, wgrads)
            assert e <= bar, (mask, path, where, e, bar)


@pytest.mark.parametrize("n", [1 << 16, 1 << 20])
def test_flux_tensor_core_at_scale_matches_generic_fp64(n):
    rng = np.random.default_rng(n % 1009)
    d, mask = 3, 0b110011
    net = _net(rng, d, 64, 4, "sin")
    X = _face_points(rng, d, mask, n // 4)
    g = _f32(rng.normal(size=n))
    want, wgrads, fam = _kernel(net, X, mask, g, "RB", 1.0, 0.4, torch.float64, "simt")
    assert fam == "simt_fma"
    got, ggrads, fam = _kernel(net, X, mask, g, "RB", 1.0, 0.4, torch.float32, "auto")
    assert fam == "tcgen05"
    assert abs(got - want) <= 1e-5 * abs(want), (got, want)
    e, where = grads_err(ggrads, wgrads)
    assert e <= 1e-5, (where, e)


def test_flux_refuses_bad_masks_before_any_launch():
    """faces == 0, faces >= 1 << 2d and a point count that is not a multiple of popcount(faces): PDE_ERR_INVALID from
    both entry points on both families, and nothing enqueued."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import _Net, ProgramSpec, NO_ENVELOPE
    lib = L.load()
    d, n = 3, 8192
    m = _net(np.random.default_rng(1), d, 64, 4, "sin").to("cuda", torch.float32)
    X = torch.rand(n, d, device="cuda") * L_BOX
    net = _Net(m, X)
    cnet = net.to_c(net.params)
    cenv = NO_ENVELOPE.to_c()
    ws = torch.empty(1 << 28, dtype=torch.uint8, device="cuda")
    row = torch.full((sum(p.numel() for p in net.params) + 2,), float("nan"), device="cuda")
    seq = torch.zeros(1, dtype=torch.int32, device="cuda")
    peers = L.Peers()
    peers.rank, peers.world = 0, 1
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    np_ = sum(p.numel() for p in net.params)
    for path in ("simt", "tc"):
        with pb.ops.kernel_path(path):
            for faces, npts in ((0, n), (1 << (2 * d), n), (0b000111, n - 1), (0b100101, 3 * 1000 + 2)):
                prog = ProgramSpec(L.PROG_FLUX, faces=faces).to_c()
                before = lib.pde_launch_count()
                rc = lib.pde_residual_loss_grad(C.byref(cnet), C.byref(cenv), C.byref(prog), X.data_ptr(), npts, None, 1.0 / npts,
                                                row.data_ptr() + (np_ + 1) * 4, row.data_ptr(), row.data_ptr() + np_ * 4,
                                                ws.data_ptr(), ws.numel(), st)
                assert rc == -1 and lib.pde_launch_count() == before, (path, faces, npts, rc)
                rc = lib.pde_residual_loss_grad_exchange(C.byref(cnet), C.byref(cenv), C.byref(prog), X.data_ptr(), npts, None,
                                                         1.0 / npts, row.data_ptr(), ws.data_ptr(), ws.numel(), C.byref(peers),
                                                         np_ + 2, seq.data_ptr(), st)
                assert rc == -1 and lib.pde_launch_count() == before, (path, faces, npts, rc)
            # the same call with a valid mask launches (and on the family asked for)
            prog = ProgramSpec(L.PROG_FLUX, faces=0b000111).to_c()
            before = lib.pde_launch_count()
            rc = lib.pde_residual_loss_grad(C.byref(cnet), C.byref(cenv), C.byref(prog), X.data_ptr(), 8190, None, 1.0 / 8190,
                                            row.data_ptr() + (np_ + 1) * 4, row.data_ptr(), row.data_ptr() + np_ * 4,
                                            ws.data_ptr(), ws.numel(), st)
            assert rc == 0 and lib.pde_launch_count() > before
            assert lib.pde_last_kernel_path() == (1 if path == "tc" else 0)
    torch.cuda.synchronize()
    assert torch.isfinite(row).all()


def _replace_faces(X, mask, per):
    X = X.clone()
    ks = [k for k in range(mask.bit_length()) if mask >> k & 1]
    for j, k in enumerate(ks):
        X[j * per:(j + 1) * per, k // 2] = L_BOX if k % 2 else 0.0
    return X


def _g_autograd(X, ks, mask):
    """s d_a u* by torch autograd of exact_u_prod_sin, in float64 at the given points."""
    import pde_b200 as pb
    Xd = X.detach().double().cpu().requires_grad_(True)
    u = pb.poisson.exact_u_prod_sin(Xd, L_BOX, ks)
    gu = torch.autograd.grad(u.sum(), Xd)[0]
    from flux_oracle import normal_derivative
    return normal_derivative(gu, mask).reshape(-1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_face_sampler_matches_interior_draw_and_manufactured_flux(dtype):
    import pde_b200 as pb
    T = pb.train
    per = 1000
    for d in range(1, 6):
        ks = [1 + (i % 2) for i in range(d)]
        for mask in sorted({(1 << 2 * d) - 1, 1 << (2 * d - 1), 0b1001 if d >= 2 else 0b10, 0b100101 if d >= 3 else 0b11}):
            nf = bin(mask).count("1")
            X, g = T.sample_faces_rhs(per, d, L_BOX, mask, ks, dtype=dtype, seed=11, offset=3)
            Xi, _, _ = T.sample_points_rhs(nf * per, d, L_BOX, None, dtype=dtype, seed=11, offset=3)
            assert X.shape == (nf * per, d)
            # the same Philox draw for every point index, the block's face coordinate replaced
            assert torch.equal(X, _replace_faces(Xi, mask, per)), (d, mask)
            want = _g_autograd(X, ks, mask)
            err = float((g.double().cpu() - want).abs().max())
            tol = 1e-12 if dtype == torch.float64 else 2e-6
            assert err <= tol * max(1.0, float(want.abs().max())), (d, mask, err)
            assert torch.allclose(g.double().cpu(), manufactured_flux(X.double().cpu(), mask, L_BOX, ks), rtol=0, atol=1e-5)
    # all faces: what the trainer's face draw gave before (one uniform draw, then the face coordinate replaced)
    fp = T._FacePoints(600, 3, L_BOX, dtype, "cuda")
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    Xf = fp.draw(5, 0, cnt).clone()
    Xi, _, _ = T.sample_points_rhs(600, 3, L_BOX, None, dtype=dtype, seed=5 ^ fp.KEY, offset=0, offset_add=cnt)
    assert torch.equal(Xf, _replace_faces(Xi, 63, 100))


def test_face_sampler_graph_replays_draw_fresh_points():
    import pde_b200 as pb
    T = pb.train
    cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    X = torch.empty(4 * 256, 2, device="cuda")
    g = torch.empty(4 * 256, device="cuda")
    T.sample_faces_rhs(256, 2, L_BOX, 0b1111, [1, 2], seed=3, offset_add=cnt, out=(X, g))   # warm-up
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        T.sample_faces_rhs(256, 2, L_BOX, 0b1111, [1, 2], seed=3, offset_add=cnt, out=(X, g))
        cnt.add_(1)
    seen = []
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        seen.append((X.clone(), g.clone()))
    assert int(cnt) == 3
    assert not torch.equal(seen[0][0], seen[1][0]) and not torch.equal(seen[1][0], seen[2][0])
    Xe, ge = T.sample_faces_rhs(256, 2, L_BOX, 0b1111, [1, 2], seed=3, offset=1)     # replay 2 used counter value 1
    assert torch.equal(Xe, seen[1][0]) and torch.equal(ge, seen[1][1])


@pytest.mark.parametrize("with_g", [True, False])
def test_boundary_loss_neumann_matches_oracle(with_g):
    import pde_b200 as pb
    d, per, mask = 3, 300, 0b011001
    torch.manual_seed(9)
    model = pb.poisson.SolutionNet(d, 32, 4, "RB").double().cuda()
    ref = copy.deepcopy(model).cpu()
    gfun = (lambda X: torch.sin(X).sum(dim=1)) if with_g else None
    torch.manual_seed(123)
    loss = pb.poisson.boundary_loss_neumann(model, L_BOX, per, d, "cuda", g=gfun, faces=mask)
    loss.backward()
    torch.manual_seed(123)      # the same torch.rand draws, in boundary_loss_dirichlet's face order
    blocks = []
    for i in range(d):
        for at_L in (False, True):
            if mask >> (2 * i + at_L) & 1:
                Xb = torch.rand(per, d, device="cuda", dtype=torch.float64) * L_BOX
                Xb[:, i] = L_BOX if at_L else 0.0
                blocks.append(Xb)
    X = torch.cat(blocks).cpu()
    g = gfun(X) if with_g else None
    want = flux_loss(ref.net, X.clone().requires_grad_(True), mask, g, L_BOX, "RB")
    want.backward()
    assert abs(float(loss.detach()) - float(want.detach())) <= 1e-10 * abs(float(want.detach()))
    got_g, want_g = _grads(model.net), _grads(ref.net)
    e, where = grads_err(got_g, want_g)
    assert e <= 1e-10, (where, e)


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("method", ["PINN", "DRM"])
def test_trainer_mixed_dirichlet_neumann_matches_reference_loop(method, graph):
    """RB model, d = 2: Neumann du/dn = du*/dn on the axis-1 faces, the soft Dirichlet penalty on the axis-0 faces.
    Five epochs equal the reference-style loop (specification losses + torch.optim.Adam, float64 on the CPU) run on the
    trainer's own face points, with g from autograd of u*."""
    import pde_b200 as pb
    torch.manual_seed(17)
    L, ks, dim, n, epochs, mask = L_BOX, [1, 2], 2, 1500, 5, 0b1100
    w = {"pde": 1.0, "bc": 50.0}
    wn = 3.0
    model = pb.poisson.SolutionNet(dim, 24, 4, "RB").double()
    ref = copy.deepcopy(model)
    model = model.cuda()
    X = torch.rand(n, dim, dtype=torch.float64) * L
    f = pb.poisson.rhs_f_for_u_sin(X, L, ks)
    tr = pb.train.FusedTrainer(model, L, ks, method=method, X=X.cuda(), f=f.cuda(), lr=2e-3, weights=w, n_boundary=400,
                               neumann_faces=mask, weight_neumann=wn, graph=graph, seed=5)
    assert tr.rows == ["pde", "bc", "neumann"] and tr.nb == 200 and tr.nn == 200
    draws, terms = [], []
    for _ in range(epochs):
        tr.step(1)
        draws.append((tr.Xb.detach().cpu().clone(), tr.Xn.detach().cpu().clone(), tr.gn.detach().cpu().clone()))
        terms.append({k: float(v) for k, v in tr.terms.items()})
    opt = torch.optim.Adam(ref.parameters(), lr=2e-3)
    from oracle import autograd_ref as AR
    for ep in range(epochs):
        Xb, Xn, gn = draws[ep]
        # the face draws: Dirichlet on faces 0, 1 (x_0 = 0, L), Neumann on faces 2, 3 (x_1 = 0, L)
        assert torch.all(Xb[:100, 0] == 0.0) and torch.all(Xb[100:, 0] == L)
        assert torch.all(Xn[:100, 1] == 0.0) and torch.all(Xn[100:, 1] == L)
        g = _g_autograd(Xn, ks, mask)
        assert float((gn - g).abs().max()) <= 1e-12
        opt.zero_grad()
        Xr = X.clone().requires_grad_(True)
        pde = (AR.pinn_loss if method == "PINN" else AR.drm_loss)(ref.net, Xr, f, L, "RB")
        bc = torch.mean(ref(Xb, L) ** 2)
        neu = flux_loss(ref.net, Xn.clone().requires_grad_(True), mask, g, L, "RB")
        total = w["pde"] * pde + w["bc"] * bc + wn * neu
        for nm, want in (("pde", pde), ("bc", bc), ("neumann", neu), ("total", total)):
            assert abs(terms[ep][nm] - float(want)) <= 1e-9 * max(1.0, abs(float(want))), (ep, nm, terms[ep][nm], float(want))
        total.backward()
        opt.step()
    for a, b in zip(model.parameters(), ref.parameters()):
        assert float((a.detach().cpu() - b.detach()).abs().max()) <= 1e-9 * max(1.0, float(b.detach().abs().max()))
    assert not torch.equal(draws[0][1], draws[1][1])


def test_trainer_neumann_refuses_fbc_model_and_bad_masks():
    import pde_b200 as pb
    m = pb.poisson.SolutionNet(2, 16, 3, "FBC").cuda()
    with pytest.raises(ValueError):
        pb.train.FusedTrainer(m, 2.0, [1, 1], n_interior=512, neumann_faces=0b0011, graph=False)
    rb = pb.poisson.SolutionNet(2, 16, 3, "RB").cuda()
    for bad in (0, 1 << 4):
        with pytest.raises(ValueError):
            pb.train.FusedTrainer(rb, 2.0, [1, 1], n_interior=512, neumann_faces=bad, graph=False)
    # pure Neumann: every face, no Dirichlet row
    tr = pb.train.FusedTrainer(rb, 2.0, [1, 1], n_interior=512, neumann_faces=0b1111, graph=False)
    assert tr.rows == ["pde", "neumann"] and not tr.use["bc"]
    tr.step(2)
    assert math.isfinite(float(tr.terms["neumann"])) and math.isfinite(float(tr.terms["total"]))


# ---------------------------------------------------------------- two or more GPUs (harness as in test_gpu_multi.py)
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _entry(rank, world, port):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        _w_trainer_neumann(rank, world)
    finally:
        dist.barrier()
        dist.destroy_process_group()


def _w_trainer_neumann(rank, world):
    """Data-parallel epoch with a Neumann row over the NVLink exchange equals the single big batch: the reference loop
    on the union of every rank's interior and face points."""
    import torch.distributed as dist
    import pde_b200 as pb
    from oracle import autograd_ref as AR
    from flux_oracle import flux_loss as FL
    L, ks, n_loc, epochs, mask = 2.0, [1, 1], 1000, 4, 0b0011
    torch.manual_seed(21)
    ref = pb.poisson.SolutionNet(2, 16, 4, "RB").double()
    X = torch.rand(n_loc * world, 2, dtype=torch.float64) * L
    f = pb.poisson.rhs_f_for_u_sin(X, L, ks)
    m = copy.deepcopy(ref).cuda()
    sl = slice(rank * n_loc, (rank + 1) * n_loc)
    tr = pb.train.FusedTrainer(m, L, ks, method="PINN", X=X[sl].cuda(), f=f[sl].cuda(), weights={"bc": 10.0}, n_boundary=200,
                               neumann_faces=mask, group=dist.group.WORLD, exchange="nvlink", lr=2e-3, seed=2)
    opt = torch.optim.Adam(ref.parameters(), lr=2e-3)
    for ep in range(epochs):
        tr.step(1)
        mine = [tr.Xb.detach().clone(), tr.Xn.detach().clone(), tr.gn.detach().clone()]
        every = []
        for t in mine:
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            every.append([p.cpu() for p in parts])
        terms = {k: float(v) for k, v in tr.terms.items()}
        opt.zero_grad()
        pde = AR.pinn_loss(ref.net, X.clone().requires_grad_(True), f, L, "RB")
        bc = torch.mean(torch.cat([ref(xb, L) for xb in every[0]]) ** 2)
        neu = sum(FL(ref.net, xn.clone().requires_grad_(True), mask, gn, L, "RB") for xn, gn in zip(every[1], every[2])) / world
        total = pde + 10.0 * bc + neu
        for nm, want in (("pde", pde), ("bc", bc), ("neumann", neu), ("total", total)):
            assert abs(terms[nm] - float(want)) <= 1e-9 * max(1.0, abs(float(want))), (ep, nm, terms[nm], float(want))
        total.backward()
        opt.step()
    for a, b in zip(m.parameters(), ref.parameters()):
        assert float((a.detach().cpu() - b.detach()).abs().max()) <= 1e-9 * max(1.0, float(b.detach().abs().max()))
    flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()])
    parts = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(parts, flat)
    assert all(torch.equal(parts[0], p) for p in parts[1:])
    tr.check()


def test_data_parallel_trainer_with_neumann_term():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_entry, args=(2, _free_port()), nprocs=2, join=True)
