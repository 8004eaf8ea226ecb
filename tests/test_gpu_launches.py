"""Launch sequences of the C ABI (run with -m gpu on a B200).

Every ABI call enqueues a fixed sequence of kernels on the caller's stream; pde_launch_count() counts them and
pde_last_kernel_path() names the kernel family that served the call.  These tests pin the number of launches of each
host path, and that a call refused for its exchange arguments enqueues nothing and leaves the caller's result row
(and the bytes past it) exactly as they were.  The ABI is driven through the ctypes structs, as in test_gpu_edges."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_gpu_edges import (ENV_POLY02, F32, F64, NQ, ORDER, PINN, POISON, SIN, _buf, _case, _dev, _envelope, _lib, _Net,
                            _path, _rand_net, _stream, _Wan, _workspace)
from oracle import jets_numpy as O

pytestmark = pytest.mark.gpu

SIMT, TC = 0, 1
PDE_ERR_INVALID = -1


def _simt_case():
    return _case(F64, 2, 3, 20, SIN, PINN, ENV_POLY02, 300, False)


def _tc_case():     # fused tensor-core kernel: fp32, 3-D, H = 64, at its 4096-point threshold
    return _case(F32, 3, 5, 64, SIN, PINN, ENV_POLY02, 4096, False)


def _split_case():  # 5-D PINN: two dimension-split passes around the pointwise residual kernel
    return _case(F32, 5, 5, 64, SIN, PINN, ENV_POLY02, 4096, False)


def _program(make, **kw):
    case = make()
    return lambda: case.run(**kw)


def _counted(call):
    """(kernels enqueued by call(), kernel family it reports)."""
    _, lib = _lib()
    before = lib.pde_launch_count()
    call()
    return lib.pde_launch_count() - before, lib.pde_last_kernel_path()


def _jets(dtype, d, H, order, N, backward):
    L, lib = _lib()
    rng = np.random.default_rng(11)
    net = _Net(*_rand_net(rng, d, H, 5, dtype), SIN, dtype)
    Ch = 1 + order * d
    X = _dev(rng.uniform(0, 2, (N, d)), dtype)
    ws = _workspace(net, order, N, 0)
    if backward:
        Jbar, g = _dev(rng.normal(size=(N, Ch)), dtype), torch.empty(net.n_params, dtype=dtype, device="cuda")
        return lambda: L.check(lib.pde_jets_backward(C.byref(net.c), order, X.data_ptr(), N, Jbar.data_ptr(), g.data_ptr(),
                                                     ws.data_ptr(), ws.numel(), _stream()), "pde_jets_backward")
    J = torch.empty(N * Ch, dtype=dtype, device="cuda")
    return lambda: L.check(lib.pde_jets_forward(C.byref(net.c), order, X.data_ptr(), N, J.data_ptr(), ws.data_ptr(),
                                                ws.numel(), _stream()), "pde_jets_forward")


def _wan():
    rng = np.random.default_rng(12)
    N, d = 1000, 2
    X = rng.uniform(-0.5, 1.5, (N, d))
    Ju, Jv = rng.normal(size=(N, 1 + d)), rng.normal(size=(N, 1 + d))
    env = _envelope(O.ENV_POLY, -0.5, 1.5, (), F32)
    prob = _Wan(F32, X, Ju, Jv, -0.5, 1.5, 0.0, rng.normal(size=N), rng.uniform(0.5, 1.5, N), 0.5, 0.75, env, env)
    return lambda: prob.run([1.0, 1.0, 1.0, 1.0], 1.0 / N, 0)


# call, kernels it enqueues, kernel family it reports (None: the call names none)
SEQUENCES = {
    "simt-program-f64": (lambda: _program(_simt_case), 3, SIMT),
    "simt-jets-forward": (lambda: _jets(F64, 2, 20, 1, 300, False), 2, SIMT),
    "simt-jets-backward": (lambda: _jets(F64, 2, 20, 1, 300, True), 3, SIMT),
    "tc-program": (lambda: _program(_tc_case), 3, TC),
    "tc-jets-forward": (lambda: _jets(F32, 3, 64, 1, 4096, False), 2, TC),
    "tc-jets-backward": (lambda: _jets(F32, 3, 64, 1, 4096, True), 3, TC),
    "split-grad": (lambda: _program(_split_case), 8, TC),
    "split-sums-dE": (lambda: _program(_split_case, grad=False), 5, TC),
    "wan-pointwise": (_wan, 2, None),
}


@pytest.mark.parametrize("name", list(SEQUENCES))
def test_launch_sequence(name):
    """pack + main kernel (+ reduction): one launch per kernel; the 5-D split adds two forward passes and the pointwise
    kernel, and with a gradient two reverse passes and a second reduction; WAN is its kernel and a finishing kernel."""
    make, launches, family = SEQUENCES[name]
    with _path("auto"):
        call = make()
        torch.cuda.synchronize()
        got, path = _counted(call)
    torch.cuda.synchronize()
    assert got == launches, f"{name}: {got} launches, expected {launches}"
    if family is not None:
        assert path == family, f"{name}: kernel family {path}, expected {family}"


@pytest.mark.parametrize("make,family", [(_simt_case, SIMT), (_tc_case, TC), (_split_case, TC)], ids=["simt", "tc", "split"])
def test_refused_exchange_enqueues_nothing(make, family):
    """pde_residual_loss_grad_exchange with a peer slot one row too short (slot_elems = n_params < n_params + 1 + K)
    is refused before anything is enqueued: no launch, and every byte of the result row and past it unchanged."""
    L, lib = _lib()
    with _path("auto"):
        case = make()
        assert case.query_path() == family
        net = case.net
        ws = _workspace(net, ORDER[case.kind], case.n, 0)
        row = net.n_params + 1 + NQ[case.kind]
        result = _buf(row, net.dtype, POISON)
        want = result.view(torch.uint8).clone()
        peer = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")   # never touched: the call is refused
        seq = torch.zeros(1, dtype=torch.int32, device="cuda")
        peers = L.Peers()
        peers.rank, peers.world = 0, 1
        peers.base[0] = peer.data_ptr()
        torch.cuda.synchronize()
        before = lib.pde_launch_count()
        rc = lib.pde_residual_loss_grad_exchange(
            C.byref(net.c), C.byref(case.env_c), C.byref(case.prog), case.Xd.data_ptr(), case.n, None, 1.0 / case.n,
            result.data_ptr(), ws.data_ptr(), ws.numel(), C.byref(peers), net.n_params, seq.data_ptr(), _stream())
        launched = lib.pde_launch_count() - before
        torch.cuda.synchronize()
    assert rc == PDE_ERR_INVALID, lib.pde_strerror(rc)
    assert launched == 0, f"{launched} kernels enqueued before the call was refused"
    assert torch.equal(result.view(torch.uint8), want), "a refused call wrote into the result row"
