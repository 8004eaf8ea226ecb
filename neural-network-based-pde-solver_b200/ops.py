"""torch.autograd bridge over the C ABI (include/pde_b200.h).

Three operators, all running on hand-written CUDA kernels:

* ``mlp_jets(model, X, order)``      network value / gradient / Hessian-diagonal channels, with a
                                      reverse sweep into the parameters (replaces ``model.net(X)`` +
                                      nested ``autograd.grad`` — Poisson_ND.py:61-71).
* ``residual_means(...)``            fused forward + envelope + residual program + reverse sweep
                                      (replaces pinn_residual_loss / drm_energy_loss + backward,
                                      Poisson_ND.py:91-103,:240 and the Schrödinger equivalents).
* ``wan_means(...)``                 two-network WAN coupling on the jets (Poisson_ND.py:105-128).

Every operator returns *means* ``m_k``; the scalar loss ``F(m_1..m_K)`` stays in Python on 0-d
tensors.  With ``group`` given, the sums (and gradient vectors) are all-reduced so that the result
equals the single big batch exactly, also for functions of means (SURVEY.md §8e).
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from dataclasses import dataclass, field
from typing import Optional, Sequence

import torch
import torch.nn as nn

from . import _lib as L

# ---------------------------------------------------------------------------------------------
# network / envelope descriptions
# ---------------------------------------------------------------------------------------------


def _linear_stack(model: nn.Module):
    """(linears, activation) of a reference-style network.

    Accepts the reference's own modules: an ``nn.Sequential`` under ``.net`` with Linear at even
    indices (Poisson_ND.py:17-23, IPW_1D_WAN.py:67-73, KH_1D.py:108-112), ``UnifiedEigenModel``
    (``.u_model.net``, KH_1D.py:216-217), a ``ModuleList`` under ``.layers``
    (QHO_1D_PINN_DRM.py:64-66) or a bare Sequential.
    """
    seq = model
    if hasattr(model, "u_model"):
        seq = model.u_model
    holder = seq   # the module that owns the activation attribute when the stack is a bare ModuleList
    for _ in range(3):   # FCN_Single.net -> FCN.layers (QHO_1D_PINN_DRM.py:85,64)
        if isinstance(seq, (nn.Sequential, nn.ModuleList)):
            break
        if hasattr(seq, "net"):
            holder = seq = seq.net
        elif hasattr(seq, "layers"):
            holder, seq = seq, seq.layers
        else:
            break
    mods = list(seq)
    linears = [m for m in mods if isinstance(m, nn.Linear)]
    others = [m for m in mods if not isinstance(m, nn.Linear)]
    if not linears:
        raise ValueError("model has no nn.Linear layers")
    act = None
    for m in others:
        name = type(m).__name__.lower()
        a = "tanh" if "tanh" in name else ("sin" if name.startswith("sin") else None)
        if a is None:
            raise NotImplementedError(f"activation {type(m).__name__} is not supported (sin / tanh only)")
        if act is not None and a != act:
            raise NotImplementedError("mixed activations are not supported")
        act = a
    if act is None:  # ModuleList of Linear only: activation kept as an attribute
        a = getattr(holder, "activation", getattr(model, "activation", None))
        name = (type(a).__name__ if a is not None else "sin").lower()
        act = "tanh" if "tanh" in name else "sin"
    return linears, act


@dataclass
class EnvelopeSpec:
    """Separable hard-constraint factor (pde_envelope)."""
    kind: int = L.ENV_NONE
    lo: float = 0.0
    hi: float = 0.0
    nodes: Sequence[Sequence[float]] = field(default_factory=list)

    def to_c(self) -> L.Envelope:
        # the ctypes struct is rebuilt only when the description changed (40 element assignments otherwise, per call)
        key = (int(self.kind), float(self.lo), float(self.hi), tuple(tuple(float(v) for v in ns) for ns in self.nodes))
        cached = getattr(self, "_c_cache", None)
        if cached is not None and cached[0] == key:
            return cached[1]
        e = self._build_c()
        object.__setattr__(self, "_c_cache", (key, e))
        return e

    def _build_c(self) -> L.Envelope:
        e = L.Envelope()
        e.kind, e.lo, e.hi = int(self.kind), float(self.lo), float(self.hi)
        for i, ns in enumerate(self.nodes):
            if len(ns) > L.MAX_NODES:
                raise NotImplementedError("too many forced nodes")
            e.n_nodes[i] = len(ns)
            for k, v in enumerate(ns):
                e.nodes[i][k] = float(v)
        return e


NO_ENVELOPE = EnvelopeSpec()


class _Net:
    """Device-side view of a model's parameters for one call."""

    def __init__(self, model: nn.Module, X: torch.Tensor):
        self.linears, act = _linear_stack(model)
        if not X.is_cuda:
            raise L.PdeError("collocation kernels run on CUDA tensors only (no CPU fallback)")
        if X.dtype not in (torch.float32, torch.float64):
            raise NotImplementedError("float32 / float64 only")
        self.dtype = X.dtype
        self.params = []
        for m in self.linears:
            if m.bias is None:
                raise NotImplementedError("Linear layers without bias are not supported")
            self.params += [m.weight, m.bias]
        for p in self.params:
            if p.device != X.device or p.dtype != X.dtype:
                raise ValueError("model parameters and points must share device and dtype")
        self.act = L.ACT_TANH if act == "tanh" else L.ACT_SIN
        self.widths = [self.linears[0].in_features] + [m.out_features for m in self.linears]
        self.dim = self.widths[0]

    def to_c(self, tensors) -> L.Net:
        n = L.Net()
        n.dtype = L.F64 if self.dtype == torch.float64 else L.F32
        n.dim, n.n_linear, n.activation = self.dim, len(self.linears), self.act
        if len(self.linears) > L.MAX_LINEAR:
            raise NotImplementedError("too many layers")
        for i, w in enumerate(self.widths):
            n.widths[i] = w
        for l in range(len(self.linears)):
            n.W[l] = tensors[2 * l].data_ptr()
            n.b[l] = tensors[2 * l + 1].data_ptr()
        return n


_WS = {}

# bench.py sets this to a list to collect (start, stop) CUDA events around each fused-kernel ABI call
KERNEL_EVENTS = None
_PATH_NAMES = {-1: "none", 0: "simt_fma", 1: "tcgen05"}


def last_kernel_path():
    """Which kernel family the last fused / jets call of this thread actually launched ("simt_fma" or
    "tcgen05"), as recorded by the library at the launch (pde_last_kernel_path)."""
    return _PATH_NAMES.get(L.load().pde_last_kernel_path(), "none")


def launch_count():
    """Kernels enqueued by libpde_b200.so in this process so far (pde_launch_count)."""
    return int(L.load().pde_launch_count())


class kernel_path:
    """Context manager forcing one kernel family: "simt", "tc" or "auto" (pde_set_kernel_path)."""
    _CODES = {"auto": -1, "simt": 0, "tc": 1}

    def __init__(self, which):
        self.code = self._CODES[which]

    def __enter__(self):
        lib = L.load()
        self.old = lib.pde_kernel_path()
        L.check(lib.pde_set_kernel_path(self.code), "pde_set_kernel_path")
        return self

    def __exit__(self, *exc):
        L.load().pde_set_kernel_path(self.old)


class _timed:
    def __init__(self, dev):
        self.on = KERNEL_EVENTS is not None
        if self.on:
            self.a, self.b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.dev = dev

    def __enter__(self):
        if self.on:
            self.a.record(torch.cuda.current_stream(self.dev))

    def __exit__(self, *exc):
        if self.on:
            self.b.record(torch.cuda.current_stream(self.dev))
            KERNEL_EVENTS.append((self.a, self.b))


def _workspace(device, nbytes):
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


_WS_NEED = {}


def _ws_for(cnet, order, n, device):
    # the size depends on the network geometry, order, point count and device only (pde_workspace_bytes is pure)
    key = (cnet.dtype, cnet.dim, cnet.n_linear, cnet.activation, tuple(cnet.widths[:cnet.n_linear + 1]), order, n,
           device.index if device.index is not None else torch.cuda.current_device(), L.load().pde_kernel_path())
    need = _WS_NEED.get(key)
    if need is None:
        val = C.c_size_t(0)
        L.check(L.load().pde_workspace_bytes(C.byref(cnet), order, n, C.byref(val)), "pde_workspace_bytes")
        need = _WS_NEED[key] = val.value
    return _workspace(device, need)


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t):
    return t.data_ptr() if t is not None else None


_unflatten = getattr(torch._C._nn, "unflatten_dense_tensors", None)


def _split_flat(flat, params):
    """Views of ``flat`` shaped like ``params``, in order (one native call where torch has it)."""
    if _unflatten is not None:
        return list(_unflatten(flat, params))
    out, o = [], 0
    for p in params:
        k = p.numel()
        out.append(flat[o:o + k].view_as(p))
        o += k
    return out


_PROG_INFO = {}


def _program_info(kind):
    """(number of quantities, derivative order) of a residual program (pure library queries, cached)."""
    info = _PROG_INFO.get(kind)
    if info is None:
        lib = L.load()
        info = _PROG_INFO[kind] = (lib.pde_program_quantities(kind), lib.pde_program_order(kind))
    return info


def _points(X):
    if X.dim() == 1:
        X = X.view(-1, 1)
    if X.dim() != 2:
        raise ValueError("points must be (N, d)")
    return X.detach().contiguous()


_EXCHANGE = {}   # process group -> comm.NvlinkAllReduce registered by use_nvlink_exchange
FUSE_EXCHANGE = True   # fold the exchange into the reduction launch (False: separate pde_allreduce_oneshot launch)


def use_nvlink_exchange(group=None, max_elems=1 << 17, dtype=torch.float32):
    """Route the exchange step of ``residual_means`` / ``wan_means`` for ``group`` through the one-kernel
    NVLink all-reduce (pde_allreduce_oneshot) instead of NCCL.  Returns the communicator."""
    from .comm import NvlinkAllReduce
    import torch.distributed as dist
    key = (group if group is not None else dist.group.WORLD, dtype)
    if key not in _EXCHANGE:
        _EXCHANGE[key] = NvlinkAllReduce(group, max_elems, dtype)
    return _EXCHANGE[key]


def _exchange_for(t, group):
    """The registered NVLink communicator that can carry ``t`` for ``group`` (None: use NCCL)."""
    if not _EXCHANGE or group is None:
        return None
    import torch.distributed as dist
    ar = _EXCHANGE.get((group if group is not None else dist.group.WORLD, t.dtype))
    if ar is not None and t.is_cuda and t.is_contiguous() and t.numel() <= ar.slot:
        return ar
    return None


def _all_reduce(t, group):
    import torch.distributed as dist
    ar = _exchange_for(t, group)
    if ar is not None:
        ar.all_reduce_(t)
    else:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


def combine_forward(buf, nparam, n_tot, group, fused):
    """Cross-rank step of a residual evaluation.  ``buf`` = [grad (nparam) | dE (1) | sums (K)] of this
    rank, the gradient part already carrying 1/N_global.  One all-reduce (the whole buffer when the
    reverse sweep was fused into the same launch, else the sums only) makes every rank hold the
    single-big-batch values; returns the means.  (SURVEY.md §8e: sums and gradient vectors are
    reduced, never per-rank losses.)"""
    sums = _row_sums(buf, nparam)
    if group is not None:
        _all_reduce(buf if fused else sums, group)
    return sums / n_tot


def combine_backward(buf, nparam, group):
    """Cross-rank step of the seeded reverse sweep (functions of means): all-reduce [grad | dE]."""
    if group is not None:
        _all_reduce(buf[:nparam + 1], group)
    return buf[:nparam], buf[nparam]


# ---------------------------------------------------------------------------------------------
# network jets
# ---------------------------------------------------------------------------------------------
class _Jets(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net: _Net, order: int, X: torch.Tensor, *params):
        lib = L.load()
        ps = [p.detach().contiguous() for p in params]
        cnet = net.to_c(ps)
        n = X.shape[0]
        Cc = 1 + order * net.dim
        J = torch.empty(n, Cc, dtype=X.dtype, device=X.device)
        ws = _ws_for(cnet, order, n, X.device)
        with torch.cuda.device(X.device):
            L.check(lib.pde_jets_forward(C.byref(cnet), order, X.data_ptr(), n, J.data_ptr(), ws.data_ptr(), ws.numel(),
                                         _stream(X.device)), "pde_jets_forward")
        ctx.net, ctx.order = net, order
        ctx.save_for_backward(X, *ps)
        return J

    @staticmethod
    def backward(ctx, Jbar):
        lib = L.load()
        X, *ps = ctx.saved_tensors
        net, order = ctx.net, ctx.order
        cnet = net.to_c(ps)
        n = X.shape[0]
        nparam = sum(p.numel() for p in ps)
        grad = torch.empty(nparam, dtype=X.dtype, device=X.device)
        Jb = Jbar.contiguous()
        ws = _ws_for(cnet, order, n, X.device)
        with torch.cuda.device(X.device):
            L.check(lib.pde_jets_backward(C.byref(cnet), order, X.data_ptr(), n, Jb.data_ptr(), grad.data_ptr(),
                                          ws.data_ptr(), ws.numel(), _stream(X.device)), "pde_jets_backward")
        grads = _split_flat(grad, ps)
        need = ctx.needs_input_grad[3:]
        return (None, None, None) + tuple(g if nd else None for g, nd in zip(grads, need))


def mlp_jets(model: nn.Module, X: torch.Tensor, order: int = 2) -> torch.Tensor:
    """(N, 1+order*d) jets of ``model.net`` at X (no envelope), differentiable w.r.t. the parameters."""
    X = _points(X)
    net = _Net(model, X)
    return _Jets.apply(net, int(order), X, *net.params)


# ---------------------------------------------------------------------------------------------
# fused residual programs
# ---------------------------------------------------------------------------------------------
@dataclass
class ProgramSpec:
    """A residual program (pde_program).  ``faces``: face mask of a ``PROG_FLUX`` batch (include/pde_b200.h: one equal
    block of points per set bit, face k = side k % 2 of axis k // 2); ignored by the other programs.  ``PROG_RITZ_VALUE``
    reads ``alpha`` as the constant g when ``f`` is None."""
    kind: int
    alpha: float = 1.0
    beta_const: float = 0.0
    energy_const: float = 0.0
    faces: int = 0

    def to_c(self, f=None, beta=None, energy=None) -> L.Program:
        """The pde_program descriptor; ``f`` / ``beta`` / ``energy``: per-point (scalar) device tensors or None."""
        p = L.Program()
        p.kind, p.alpha, p.beta_const, p.energy_const = self.kind, self.alpha, self.beta_const, self.energy_const
        p.faces = int(self.faces)
        p.f, p.beta, p.energy = _ptr(f), _ptr(beta), _ptr(energy)
        return p


_MSE = ProgramSpec(L.PROG_MSE)


def _row_sums(row, nparam):
    """The sums of a [grad (nparam) | dE (1) | sums (K)] row."""
    return row[nparam + 1:]


def _residual_row(cnet, cenv, prog, X, n, inv_n, ws, row, nparam, seed=None, sums=None, want_grad=True, ar=None):
    """One residual-program launch into ``row`` = [grad (nparam) | dE (1) | sums (K)] (1-D, contiguous): the layout
    that pde_residual_loss_grad writes and that the all-reduce and pde_residual_loss_grad_exchange carry.

    ``seed``: device cotangents of the means (seeded reverse sweep); ``sums``: write the sums there instead of into
    the row; ``want_grad=False``: sums only (``row`` may then be None); ``ar``: an ``NvlinkAllReduce`` whose exchange
    of the whole row is folded into the reduction launch."""
    lib, st = L.load(), _stream(X.device)
    if ar is not None:
        L.check(lib.pde_residual_loss_grad_exchange(C.byref(cnet), C.byref(cenv), C.byref(prog), X.data_ptr(), n,
                                                    _ptr(seed), inv_n, row.data_ptr(), ws.data_ptr(), ws.numel(),
                                                    C.byref(ar.peers), ar.slot, ar.seq.data_ptr(), st),
                "pde_residual_loss_grad_exchange")
        return
    es = X.element_size()
    gptr = row.data_ptr() if want_grad else None
    sptr = sums.data_ptr() if sums is not None else row.data_ptr() + (nparam + 1) * es
    L.check(lib.pde_residual_loss_grad(C.byref(cnet), C.byref(cenv), C.byref(prog), X.data_ptr(), n, _ptr(seed), inv_n,
                                       sptr, gptr, gptr + nparam * es if want_grad else None, ws.data_ptr(), ws.numel(),
                                       st), "pde_residual_loss_grad")


class _Residual(torch.autograd.Function):
    """means[K] of a residual program; backward = sum_k gbar_k * d(mean_k)/d(theta, E)."""

    @staticmethod
    def forward(ctx, net, env, spec, group, n_global, need_grad, X, f, beta, energy, *params):
        ps = [p.detach().contiguous() for p in params]
        cnet = net.to_c(ps)
        n = X.shape[0]
        K, order = _program_info(spec.kind)
        dev, dt = X.device, X.dtype
        nparam = sum(p.numel() for p in ps)
        n_tot = float(n if n_global is None else n_global)
        ctx.cfg = (net, env, spec, group, n_tot)
        ctx.K = K
        fused = (K == 1) and need_grad
        # one buffer [grad (nparam) | dE (1) | sums (K)] so that one all-reduce covers everything
        buf = torch.zeros(nparam + 1 + K, dtype=dt, device=dev)
        e_dev = energy.detach().reshape(1).to(dt) if energy is not None else None
        prog, cenv = spec.to_c(f, beta, e_dev), env.to_c()
        ws = _ws_for(cnet, order, n, dev)
        # exchange folded into the reduction of the per-CTA partials: no separate all-reduce launch
        ar = _exchange_for(buf, group) if (fused and FUSE_EXCHANGE) else None
        with torch.cuda.device(dev), _timed(dev):
            _residual_row(cnet, cenv, prog, X, n, 1.0 / n_tot, ws, buf, nparam, want_grad=fused, ar=ar)
        means = combine_forward(buf, nparam, n_tot, None if ar is not None else group, fused)
        ctx.fused = fused
        ctx.has_energy = energy is not None
        if fused:
            ctx.save_for_backward(buf)
            ctx.ps = ps
        else:
            ctx.save_for_backward(X, f, beta, e_dev, *ps)
        return means     # (a fresh tensor: the division in combine_forward)

    @staticmethod
    def backward(ctx, gmeans):
        net, env, spec, group, n_tot = ctx.cfg
        n_in = 10
        if ctx.fused:
            (buf,) = ctx.saved_tensors
            nparam = buf.numel() - 1 - ctx.K
            flat = buf[:nparam] * gmeans          # (K = 1: gmeans has one element)
            gE = (buf[nparam] * gmeans[0]) if ctx.has_energy else None
            grads = _split_flat(flat, ctx.ps)
        else:
            X, f, beta, e_dev, *ps = ctx.saved_tensors
            cnet = net.to_c(ps)
            n = X.shape[0]
            dev, dt = X.device, X.dtype
            nparam = sum(p.numel() for p in ps)
            buf = torch.zeros(nparam + 1 + ctx.K, dtype=dt, device=dev)
            seed = gmeans.detach().to(dt).contiguous()
            ws = _ws_for(cnet, _program_info(spec.kind)[1], n, dev)
            with torch.cuda.device(dev):
                _residual_row(cnet, env.to_c(), spec.to_c(f, beta, e_dev), X, n, 1.0 / n_tot, ws, buf, nparam, seed=seed)
            flat, dE = combine_backward(buf, nparam, group)
            grads = _split_flat(flat, ps)
            gE = dE if ctx.has_energy else None
        need = ctx.needs_input_grad
        out = [None] * n_in
        if gE is not None and need[9]:
            out[9] = gE.reshape(())
        out += [g if nd else None for g, nd in zip(grads, need[n_in:])]
        return tuple(out)


def _global_count(n, group, n_global):
    """Points of the global batch: with ``group`` and no explicit ``n_global`` every rank is taken to hold ``n``
    points (dividing the all-reduced sums by the local count would make loss and gradient world times too large)."""
    if n_global is not None or group is None:
        return n_global
    import torch.distributed as dist
    return n * dist.get_world_size(group)


def _coefficients(spec, X, f, beta, energy):
    """(spec, f, beta, energy) of one call: a float ``beta`` / ``energy`` folded into the spec's constants, per-point
    ``f`` / ``beta`` as flat contiguous tensors of the points' dtype with one value per point, a tensor ``energy`` as
    given.  Already conforming coefficients are passed through without a copy."""
    def coef(t):
        if t is None:
            return None
        t = t.detach()
        if t.dtype != X.dtype:
            t = t.to(X.dtype)
        t = t.reshape(-1)
        if not t.is_contiguous():
            t = t.contiguous()
        if t.numel() != X.shape[0] or t.device != X.device:
            raise ValueError("per-point coefficient must have one value per point on the points' device")
        return t

    if energy is not None and not torch.is_tensor(energy):
        spec, energy = dataclasses.replace(spec, energy_const=float(energy)), None
    if beta is not None and not torch.is_tensor(beta):
        spec, beta = dataclasses.replace(spec, beta_const=float(beta)), None
    return spec, coef(f), coef(beta), energy


def residual_means(model, X, spec: ProgramSpec, env: EnvelopeSpec = NO_ENVELOPE, f=None, beta=None, energy=None,
                   group=None, n_global: Optional[int] = None) -> torch.Tensor:
    """Means of the program's per-point quantities, differentiable w.r.t. the network parameters
    (and the scalar ``energy`` when it is a tensor that requires grad)."""
    X = _points(X)
    net = _Net(model, X)
    n_global = _global_count(X.shape[0], group, n_global)
    spec, f, beta, e = _coefficients(spec, X, f, beta, energy)
    # (grad mode is off inside Function.forward, so decide here whether the fused reverse sweep runs)
    need_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in net.params) or
                                             (e is not None and e.requires_grad))
    return _Residual.apply(net, env, spec, group, n_global, need_grad, X, f, beta, e, *net.params)


def residual_mean(model, X, spec: ProgramSpec, env: EnvelopeSpec = NO_ENVELOPE, **kw) -> torch.Tensor:
    """``residual_means`` of a one-quantity program (PINN residual, Deep Ritz energy, MSE) as a 0-d tensor.  A view:
    indexing ``means[0]`` costs two launches in backward (select_backward = zero fill + copy), a reshape none."""
    m = residual_means(model, X, spec, env, **kw)
    if m.numel() != 1:
        raise ValueError("residual_mean is for programs with one quantity")
    return m.reshape(())


# ---------------------------------------------------------------------------------------------
# WAN coupling of two networks
# ---------------------------------------------------------------------------------------------
@dataclass
class WanSpec:
    alpha: float = 1.0
    beta_const: float = 0.0
    energy_const: float = 0.0
    w_lo: float = 0.0
    w_hi: float = 2.0
    eps_den: float = 0.0

    def to_c(self, dtype, dim, env_u, env_v, f=None, beta=None, energy=None) -> L.Wan:
        """The pde_wan descriptor for points of ``dtype`` / ``dim``; ``f`` / ``beta`` / ``energy``: per-point (scalar)
        device tensors or None."""
        w = L.Wan()
        w.dtype = L.F64 if dtype == torch.float64 else L.F32
        w.dim = dim
        w.alpha, w.beta_const, w.energy_const = self.alpha, self.beta_const, self.energy_const
        w.w_lo, w.w_hi, w.eps_den = self.w_lo, self.w_hi, self.eps_den
        w.f, w.beta, w.energy = _ptr(f), _ptr(beta), _ptr(energy)
        w.env_u, w.env_v = env_u.to_c(), env_v.to_c()
        return w


class _WanPoint(torch.autograd.Function):
    """means[4] (+ d mean0/dE) from the two networks' jets; backward produces jet cotangents."""

    @staticmethod
    def forward(ctx, spec, env_u, env_v, group, n_global, X, f, beta, energy, Ju, Jv):
        lib = L.load()
        n, d = X.shape
        dev, dt = X.device, X.dtype
        n_tot = float(n if n_global is None else n_global)
        e_dev = energy.detach().reshape(1).to(dt) if energy is not None else None
        w = spec.to_c(dt, d, env_u, env_v, f, beta, e_dev)
        sums = torch.empty(5, dtype=dt, device=dev)    # all five written by the launch (wan_finish_kernel)
        ws = _workspace(dev, 1 << 20)
        Juc, Jvc = Ju.detach().contiguous(), Jv.detach().contiguous()
        with torch.cuda.device(dev):
            L.check(lib.pde_wan_pointwise(C.byref(w), X.data_ptr(), n, Juc.data_ptr(), Jvc.data_ptr(), None, 1.0 / n_tot,
                                          sums.data_ptr(), None, None, ws.data_ptr(), ws.numel(), _stream(dev)),
                    "pde_wan_pointwise")
        if group is not None:
            _all_reduce(sums, group)
        ctx.cfg = (spec, env_u, env_v, n_tot)
        ctx.has_energy = energy is not None
        ctx.save_for_backward(X, f, beta, e_dev, Juc, Jvc, sums)
        return sums[:4] / n_tot

    @staticmethod
    def backward(ctx, gmeans):
        lib = L.load()
        spec, env_u, env_v, n_tot = ctx.cfg
        X, f, beta, e_dev, Ju, Jv, sums = ctx.saved_tensors
        n, d = X.shape
        dev, dt = X.device, X.dtype
        w = spec.to_c(dt, d, env_u, env_v, f, beta, e_dev)
        seed = gmeans.detach().to(dt).contiguous()
        Jbu, Jbv = torch.empty_like(Ju), torch.empty_like(Jv)
        scratch = torch.empty(5, dtype=dt, device=dev)
        ws = _workspace(dev, 1 << 20)
        with torch.cuda.device(dev):
            L.check(lib.pde_wan_pointwise(C.byref(w), X.data_ptr(), n, Ju.data_ptr(), Jv.data_ptr(), seed.data_ptr(),
                                          1.0 / n_tot, scratch.data_ptr(), Jbu.data_ptr(), Jbv.data_ptr(), ws.data_ptr(),
                                          ws.numel(), _stream(dev)), "pde_wan_pointwise")
        gE = None
        if ctx.has_energy and ctx.needs_input_grad[8]:
            gE = (sums[4] / n_tot * gmeans[0]).reshape(())   # sums already all-reduced in forward
        need = ctx.needs_input_grad
        return (None, None, None, None, None, None, None, None, gE, Jbu if need[9] else None, Jbv if need[10] else None)


def wan_means(u_model, v_model, X, spec: WanSpec, env_u=NO_ENVELOPE, env_v=NO_ENVELOPE, f=None, beta=None, energy=None,
              group=None, n_global=None, u_jets=None, v_jets=None):
    """means (q0..q3) of the WAN weak-form quantities for the u / v networks (pde_wan_pointwise).

    The jets of both networks come from the fused network kernels; parameters with
    ``requires_grad=False`` (the reference toggles them, IPW_1D_WAN.py:186-200) get no gradient.
    With ``group`` the per-rank parameter gradients are averaged exactly because the means are
    all-reduced before ``F`` is applied and the cotangents carry 1/N_global.

    ``u_jets`` / ``v_jets``: order-1 jets of a *frozen* network on the same points (``frozen_jets``),
    reused instead of re-evaluating that network — the critic steps of the minimax loop run on fixed
    points with the other network's parameters switched off (IPW_1D_WAN.py:186-194, KH_1D.py:343-352).
    """
    X = _points(X)
    n_global = _global_count(X.shape[0], group, n_global)
    spec, f, beta, e = _coefficients(spec, X, f, beta, energy)
    Ju = mlp_jets(u_model, X, 1) if u_jets is None else _check_jets(u_jets, X)
    Jv = mlp_jets(v_model, X, 1) if v_jets is None else _check_jets(v_jets, X)
    return _WanPoint.apply(spec, env_u, env_v, group, n_global, X, f, beta, e, Ju, Jv)


class _WanScalars(torch.autograd.Function):
    """(loss_pde, loss_v, loss_norm, total) of the four WAN means in one launch (pde_wan_scalars); backward = J^T g."""

    @staticmethod
    def forward(ctx, means, kind, consts):
        lib = L.load()
        dev, dt = means.device, means.dtype
        m = means.detach().contiguous()
        out = torch.empty(4, dtype=dt, device=dev)
        jac = torch.empty(4, 4, dtype=dt, device=dev)
        carr = (C.c_double * 6)(*[float(c) for c in consts])
        with torch.cuda.device(dev):
            L.check(lib.pde_wan_scalars(L.F64 if dt == torch.float64 else L.F32, int(kind), m.data_ptr(), carr, out.data_ptr(),
                                        jac.data_ptr(), _stream(dev)), "pde_wan_scalars")
        ctx.save_for_backward(jac)
        ctx.set_materialize_grads(False)
        return out[0], out[1], out[2], out[3]

    @staticmethod
    def backward(ctx, *gouts):
        (jac,) = ctx.saved_tensors
        gm = None
        for k, g in enumerate(gouts):
            if g is not None:
                t = jac[k] * g
                gm = t if gm is None else gm + t
        return gm, None, None


def wan_scalar_losses(means, *, kind=0, eps_pde=1e-8, eps_log=1e-8, vol=1.0, reg=0.0, w_pde=1.0, w_norm=1.0):
    """(loss_pde, loss_v, loss_norm, total) from the means of ``wan_means`` — the scalar end of every reference
    WAN_loss (Poisson_ND.py:118-127, IPW_1D_WAN.py:108-114, QHO_2D.py:218-224, KH_1D.py:263-268) as one launch
    instead of ~25 zero-dimensional tensor operations."""
    return _WanScalars.apply(means, kind, (eps_pde, eps_log, vol, reg, w_pde, w_norm))


def _check_jets(J, X):
    if J.shape != (X.shape[0], 1 + X.shape[1]) or J.dtype != X.dtype or J.device != X.device:
        raise ValueError("frozen jets must be the (N, 1+d) order-1 jets of the same points")
    return J.detach()


def frozen_jets(model, X, order: int = 1):
    """Jets of a network whose parameters are not being trained in this phase: one forward launch,
    no autograd node.  Pass the result as ``u_jets`` / ``v_jets`` to the WAN losses for as long as
    neither the points nor that network change (SURVEY.md §8f-2)."""
    with torch.no_grad():
        return mlp_jets(model, X, order).detach()


def all_reduce_grads(params, group=None):
    """Sum ``p.grad`` over ranks (used with wan_means, whose network sweeps are rank local)."""
    import torch.distributed as dist
    gs = [p.grad for p in params if p.grad is not None]
    if not gs:
        return
    flat = torch.cat([g.reshape(-1) for g in gs])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    for g, r in zip(gs, _split_flat(flat, gs)):
        g.copy_(r)
