"""GPU tests of the parabolic program (PDE_PROG_PARABOLIC): both kernel families against the float64 autograd
specification (tests/heat_oracle.py), 2^20 points on the automatic path against the float64 generic kernel, boxes of
every size, the heat drop-in, its launch count and workspace, the convergence bound of tools/heat_convergence.py and the
folded multi-GPU exchange.

Bars (DESIGN.md §7): float64 on the generic kernel 1e-10; float32 max(1e-5, 2 e32), e32 being the distance between the
specification run in float32 and in float64 on the same inputs (and on inputs one float32 ulp away)."""
import copy
import ctypes as C
import functools
import math
import os
import socket
import sys

import numpy as np
import pytest
import torch

from conftest import grads_err
from heat_oracle import parabolic_loss
from test_gpu_neumann import _f32, _grads, _Holder, _net

pytestmark = pytest.mark.gpu
N = 4096
FAMILY = {"tc": "tcgen05", "simt": "simt_fma", "simt64": "simt_fma"}


def _coefs(rng, case, n):
    """(alpha, beta, E, f) of a case: 'a' per-point beta, f given, trainable E; 'b' constant beta and E, f NULL."""
    if case == "a":
        return -0.3, _f32(rng.uniform(0.5, 1.5, n)), 0.25, _f32(rng.normal(size=n))
    return -0.3, 0.7, 0.2, None


def _oracle(net, X, alpha, beta, E, f, dtype=torch.float64):
    """(loss, grads, dloss/dE) of the specification on the CPU in ``dtype``."""
    ref = copy.deepcopy(net).to(dtype)
    Xt = torch.tensor(X, dtype=dtype).requires_grad_(True)
    bt = torch.tensor(beta, dtype=dtype) if isinstance(beta, np.ndarray) else beta
    ft = None if f is None else torch.tensor(f, dtype=dtype)
    Et = torch.tensor(E, dtype=dtype, requires_grad=True)
    loss = parabolic_loss(ref, Xt, ft, alpha, bt, Et)
    loss.backward()
    return float(loss.detach()), _grads(ref), float(Et.grad)


@functools.lru_cache(maxsize=None)
def _case(d, act, case, seed=0):
    rng = np.random.default_rng(100 * d + 10 * (act == "tanh") + (case == "b") + seed)
    net = _net(rng, d, 64, 4, act)
    X = _f32(rng.uniform(0.0, 2.0, (N, d)))
    return (net, X) + _coefs(rng, case, N)


@functools.lru_cache(maxsize=None)
def _e32(d, act, case):
    return _e32_of(*_case(d, act, case))


def _e32_of(net, X, alpha, beta, E, f, draws=8):
    """The specification's own float32 error (loss, gradients, dE) over these inputs and eight inputs one float32 ulp
    away (the rule of test_gpu_neumann.py)."""
    gen = np.random.default_rng(7)
    worst = 0.0
    for k in range(draws + 1):
        jit = (lambda t: t * (1.0 + gen.uniform(-1, 1, np.shape(t)) * 2.0 ** -24)) if k else (lambda t: t)
        netj = copy.deepcopy(net)
        if k:
            with torch.no_grad():
                for p in netj.parameters():
                    p.copy_(torch.tensor(jit(p.detach().numpy())))
        bj = jit(beta) if isinstance(beta, np.ndarray) else beta
        args = (jit(X), alpha, bj, E, None if f is None else jit(f))
        l32, g32, e32 = _oracle(netj, *args, dtype=torch.float32)
        l64, g64, e64 = _oracle(netj, *args)
        worst = max(worst, abs(l32 - l64) / max(abs(l64), 1e-3), grads_err(g32, g64)[0],
                    abs(e32 - e64) / max(abs(e64), 1e-3))
    return worst


def _kernel(net, X, alpha, beta, E, f, dtype, path, energy_tensor=True):
    """loss, gradients and dloss/dE of the PARABOLIC program through ops.residual_means on the given kernel family."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import NO_ENVELOPE, ProgramSpec, residual_means
    m = copy.deepcopy(net).to("cuda", dtype)
    dev = lambda a: None if a is None else torch.tensor(a, dtype=dtype, device="cuda")
    Xg = dev(X)
    spec = ProgramSpec(L.PROG_PARABOLIC, alpha)
    bg = dev(beta) if isinstance(beta, np.ndarray) else float(beta)
    Eg = torch.tensor(E, dtype=dtype, device="cuda", requires_grad=True) if energy_tensor else float(E)
    with pb.ops.kernel_path("simt" if path == "simt64" else path):
        loss = residual_means(_Holder(m, "RB"), Xg, spec, NO_ENVELOPE, f=dev(f), beta=bg, energy=Eg)[0]
        loss.backward()
        family = pb.ops.last_kernel_path()
    dE = float(Eg.grad) if energy_tensor else None
    return float(loss.detach()), _grads(m), dE, family


def _check(got, want, bar, what):
    (l, g, dE), (lw, gw, dEw) = got, want
    assert abs(l - lw) <= bar * max(abs(lw), 1e-3), (what, "loss", l, lw)
    err, where = grads_err(g, gw)
    assert err <= bar, (what, err, where)
    if dE is not None:
        assert abs(dE - dEw) <= bar * max(abs(dEw), 1e-3), (what, "dE", dE, dEw)


def _bar(path, d, act, case):
    return 1e-10 if path == "simt64" else max(1e-5, 2.0 * _e32(d, act, case))


@pytest.mark.parametrize("case", ["a", "b"])
@pytest.mark.parametrize("act", ["sin", "tanh"])
@pytest.mark.parametrize("path", ["tc", "simt", "simt64"])
@pytest.mark.parametrize("d", [2, 3, 4])
def test_parabolic_program_matches_the_specification(d, path, act, case):
    net, X, alpha, beta, E, f = _case(d, act, case)
    want = _oracle(net, X, alpha, beta, E, f)
    l, g, dE, family = _kernel(net, X, alpha, beta, E, f, torch.float64 if path == "simt64" else torch.float32, path,
                               energy_tensor=(case == "a"))
    assert family == FAMILY[path]
    _check((l, g, dE), want, _bar(path, d, act, case), f"d{d} {path} {act} {case}")


@pytest.mark.parametrize("case", ["a", "b"])
@pytest.mark.parametrize("path", ["simt", "simt64"])
def test_five_dimensional_parabolic_runs_on_the_generic_kernel(path, case):
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import ProgramSpec, _Net
    net, X, alpha, beta, E, f = _case(5, "sin", case)
    want = _oracle(net, X, alpha, beta, E, f)
    got = _kernel(net, X, alpha, beta, E, f, torch.float64 if path == "simt64" else torch.float32, path,
                  energy_tensor=(case == "a"))
    assert got[3] == "simt_fma"
    _check(got[:3], want, _bar(path, 5, "sin", case), f"d5 {path} {case}")
    # the query agrees: the 5-D split serves PINN only, so the automatic and the forced path answer 0 for PARABOLIC
    m = copy.deepcopy(net).to("cuda", torch.float32)
    Xg = torch.tensor(X, dtype=torch.float32, device="cuda")
    cn = _Net(m, Xg).to_c([p.detach() for p in m.parameters()])
    lib = L.load()
    for which in ("auto", "tc"):
        with pb.ops.kernel_path(which):
            assert lib.pde_query_path(C.byref(cn), C.byref(ProgramSpec(L.PROG_PARABOLIC, alpha).to_c()), 1 << 20) == 0
            assert lib.pde_query_path(C.byref(cn), C.byref(ProgramSpec(L.PROG_PINN, alpha).to_c()), 1 << 20) == 1


def test_2_20_points_on_the_automatic_path():
    """d = 4 at 2^20 points: the automatic path is the tensor-core kernel, within 1e-5 of the float64 generic kernel."""
    rng = np.random.default_rng(5)
    n = 1 << 20
    net = _net(rng, 4, 64, 5, "sin")
    X = _f32(rng.uniform(0.0, 2.0, (n, 4)))
    beta, f = _f32(rng.uniform(0.5, 1.5, n)), _f32(rng.normal(size=n))
    got = _kernel(net, X, -0.3, beta, 0.25, f, torch.float32, "auto")
    assert got[3] == "tcgen05"
    want = _kernel(net, X, -0.3, beta, 0.25, f, torch.float64, "simt64")
    _check(got[:3], want[:3], 1e-5, "2^20 d4")


BOXES = [1 / 32, 1.0, 60.0, 200.0]


@pytest.mark.parametrize("path", ["tc", "simt"])
@pytest.mark.parametrize("L_box", BOXES)
def test_box_sizes(L_box, path):
    """W0 scaled by p = 2^round(log2(2 / L)) and points in [0, L]^3 (the rule of test_gpu_tc_scaling.py): u_t ~ p and
    Lap_x u ~ p^2, so alpha = -1 / p, beta and f carry p, and every term of the residual is O(p).  f is one-signed:
    with a random-sign f dominating r, the output-bias gradient mean(2 r (beta - E)) would be a cancelling sum whatever
    the kernel."""
    p = 2.0 ** round(math.log2(2.0 / L_box))
    rng = np.random.default_rng(int(L_box * 64))
    net = _net(rng, 3, 64, 5, "sin")
    with torch.no_grad():
        net[0].weight.mul_(p)
    X = _f32(rng.uniform(0.0, L_box, (N, 3)))
    beta, f = _f32(p * rng.uniform(0.5, 1.5, N)), _f32(p * rng.uniform(0.5, 1.5, N))
    alpha = -1.0 / p
    want = _oracle(net, X, alpha, beta, 0.0, f)
    got = _kernel(net, X, alpha, beta, 0.0, f, torch.float32, path, energy_tensor=False)
    assert got[3] == FAMILY[path]
    _check(got[:3], want, max(1e-5, 2.0 * _e32_of(net, X, alpha, beta, 0.0, f)), f"L={L_box} {path}")


def test_heat_drop_in_matches_the_specification():
    import pde_b200 as pb
    rng = np.random.default_rng(11)
    net = _net(rng, 3, 64, 5, "sin")
    X = _f32(rng.uniform(0.0, 1.0, (8192, 3)))
    f = _f32(rng.uniform(0.5, 1.5, 8192))   # one-signed, as in test_box_sizes: no cancelling gradient sums
    kappa = 0.4
    want = _oracle(net, X, -kappa, 0.0, 0.0, f)
    m = copy.deepcopy(net).to("cuda", torch.float32)
    loss = pb.heat.heat_residual_loss(_Holder(m, "RB"), torch.tensor(X, dtype=torch.float32, device="cuda"),
                                      torch.tensor(f, dtype=torch.float32, device="cuda"), kappa)
    loss.backward()
    assert pb.ops.last_kernel_path() == "tcgen05"
    bar = max(1e-5, 2.0 * _e32_of(net, X, -kappa, 0.0, 0.0, f))
    _check((float(loss.detach()), _grads(m), None), want, bar, "heat_residual_loss")


@pytest.mark.parametrize("path", ["tc", "simt"])
def test_launches_and_workspace_equal_the_pinn_step(path):
    """A parabolic call enqueues as many kernels as a PINN call at the same shape, and runs in exactly the workspace
    pde_workspace_bytes(net, 2, n) gives."""
    import pde_b200 as pb
    from pde_b200 import _lib as L
    from pde_b200.ops import ProgramSpec, _Net
    n = 8192
    torch.manual_seed(2)
    m = pb.poisson.SolutionNet(3, 64, 5, "RB").cuda()
    X = torch.rand(n, 3, device="cuda")
    f = torch.randn(n, device="cuda")
    params = [p.detach() for p in m.parameters()]
    cn = _Net(m, X).to_c(params)
    lib = L.load()
    ws = C.c_size_t(0)
    L.check(lib.pde_workspace_bytes(C.byref(cn), 2, n, C.byref(ws)), "pde_workspace_bytes")
    nparam = sum(p.numel() for p in params)
    buf = torch.empty(ws.value + 256, dtype=torch.uint8, device="cuda")
    base = (buf.data_ptr() + 255) // 256 * 256
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {}
    with pb.ops.kernel_path(path):
        for kind in (L.PROG_PINN, L.PROG_PARABOLIC):
            prog = ProgramSpec(kind, -0.5).to_c(f=f)
            sums = torch.zeros(1, device="cuda")
            grad = torch.zeros(nparam, device="cuda")
            torch.cuda.synchronize()
            c0 = lib.pde_launch_count()
            rc = lib.pde_residual_loss_grad(C.byref(cn), None, C.byref(prog), X.data_ptr(), n, None, 1.0 / n,
                                            sums.data_ptr(), grad.data_ptr(), None, base, ws.value, stream)
            assert rc == 0, (kind, rc)
            out[kind] = lib.pde_launch_count() - c0
            assert pb.ops.last_kernel_path() == FAMILY[path]
            torch.cuda.synchronize()
            if kind == L.PROG_PARABOLIC:
                want = float(pb.heat.heat_residual_loss(m, X, f, 0.5).detach())
                assert abs(float(sums) / n - want) <= 1e-5 * abs(want)
    assert out[L.PROG_PARABOLIC] == out[L.PROG_PINN], out


# ---------------------------------------------------------------- convergence (tools/heat_convergence.py)
# profiles/heat_convergence.json (B200): the best relative L2 error of the checkpoints at 500, 1000 and 1500 epochs is
# 1.75e-2 (4.3e-3 after 4500); the bound leaves ~3x for run-to-run differences of the training
CONV_EPOCHS = 1500
CONV_BOUND = 0.05


def test_heat_convergence_short_run():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import heat_convergence as HC
    _, rec = HC.run(CONV_EPOCHS, every=500, seed=0)
    assert rec["kernel_path"] == "tcgen05"
    assert rec["best_l2"] <= CONV_BOUND, rec


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
    """heat_residual_loss with group= and the exchange folded into the NVLink reduction equals the single big batch."""
    import torch.distributed as dist
    import pde_b200 as pb
    n_loc = 6000
    torch.manual_seed(3)
    m = pb.poisson.SolutionNet(3, 64, 5, "RB").cuda()
    X = torch.rand(n_loc * world, 3, device="cuda")
    f = torch.cos(X).sum(dim=1)
    sl = slice(rank * n_loc, (rank + 1) * n_loc)
    pb.ops.use_nvlink_exchange(None, 1 << 15, torch.float32)
    m.zero_grad()
    big = pb.heat.heat_residual_loss(m, X, f, 0.3)
    big.backward()
    want = [p.grad.clone() for p in m.parameters()]
    m.zero_grad()
    part = pb.heat.heat_residual_loss(m, X[sl], f[sl], 0.3, group=dist.group.WORLD)
    part.backward()
    assert pb.ops.last_kernel_path() == "tcgen05"
    assert abs(float(part) - float(big)) <= 2e-6 * max(abs(float(big)), 1e-3), (float(part), float(big))
    for p, w in zip(m.parameters(), want):
        assert float((p.grad - w).abs().max()) <= 1e-5 * float(w.abs().max())
    pb.ops._EXCHANGE[(dist.group.WORLD, torch.float32)].check()


def test_heat_folded_exchange_matches_single_batch():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_entry, args=(2, _free_port()), nprocs=2, join=True)
