"""Fused training epoch around the loss step (SURVEY.md §8f-1, §8f-3).

``train_poisson_nd`` (Poisson_ND.py:215-300) spends an epoch on: [draw points, evaluate f] -> loss ->
``loss.backward()`` -> ``Adam.step()`` -> draw test points -> L2 error -> ``.item()`` -> keep the best
state on the CPU.  Here the same epoch is a fixed sequence of launches on one stream —

    pde_sample_points_rhs  (optional, when points are redrawn every epoch)
    pde_residual_loss_grad (the fused tcgen05 / SIMT loss step: sums, flat gradient)
    pde_sample_faces_rhs + pde_residual_loss_grad per boundary term (Dirichlet penalty, Neumann flux), data / norm terms
    all-reduce of [grad | dE | sums]  (only with ``group``)
    pde_adam_step          (fused Adam on the flat gradient, parameters updated in place)
    pde_sample_points_rhs + pde_residual_loss_grad(value only) + pde_keep_best  (optional evaluation)

— captured once into a CUDA graph and replayed; nothing is read back to the host unless the caller
asks for ``loss`` / ``l2``.  Sampling is statistically, not bitwise, equivalent to ``torch.rand``
(Philox4x32-10 keyed by seed, counter = point index and epoch); everything else follows the
reference's arithmetic (Adam: torch.optim.Adam defaults, single-tensor formula).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence

import torch

from . import _lib as L
from .ops import _MSE, EnvelopeSpec, ProgramSpec, _Net, _residual_row, _row_sums, _split_flat, _stream, _ws_for


def sample_points_rhs(n, dim, L_box, ks=None, *, dtype=torch.float32, device="cuda", seed=0, offset=0, lo=0.0,
                      want_u=False, want_f=True, X=None, offset_add=None, out=None):
    """(X, u_exact, f): uniform points in [lo, L_box)^dim (or the given ``X``) with the manufactured
    solution / right-hand side of Poisson_ND.py:49-58 evaluated in the same launch.  ``offset`` selects the
    Philox counter block: draws with different offsets are independent (epoch number; ``rank_offset(r)`` for the
    ranks of a data-parallel run).  ``offset_add``: device int64 scalar added to ``offset`` at run time (a draw
    counter, so that a replayed CUDA graph draws fresh points); ``out=(X, u, f)``: write into existing tensors."""
    lib = L.load()
    dev = torch.device(device)
    if X is not None:
        Xin = X.detach().contiguous()
        n, dim, dtype, dev = Xin.shape[0], Xin.shape[1], Xin.dtype, Xin.device
        Xout = Xin
    else:
        Xin = None
        Xout = out[0] if out is not None else torch.empty(n, dim, dtype=dtype, device=dev)
    if out is not None:
        u, f = out[1], out[2]
    else:
        u = torch.empty(n, 1, dtype=dtype, device=dev) if (want_u and ks is not None) else None
        f = torch.empty(n, 1, dtype=dtype, device=dev) if (want_f and ks is not None) else None
    karr = (C.c_double * dim)(*[float(k) for k in ks]) if ks is not None else None
    with torch.cuda.device(dev):
        L.check(lib.pde_sample_points_rhs(L.F64 if dtype == torch.float64 else L.F32, dim, n, float(lo), float(L_box),
                                          int(seed), int(offset), offset_add.data_ptr() if offset_add is not None else None,
                                          karr, float(L_box),
                                          Xin.data_ptr() if Xin is not None else None,
                                          None if Xin is not None else Xout.data_ptr(),
                                          u.data_ptr() if u is not None else None,
                                          f.data_ptr() if f is not None else None, _stream(dev)),
                "pde_sample_points_rhs")
    return Xout, u, f


def all_faces(dim):
    """The face mask with every face of [lo, hi]^dim set (include/pde_b200.h: face k = side k % 2 of axis k // 2)."""
    return (1 << (2 * int(dim))) - 1


def sample_faces_rhs(n_per_face, dim, L_box, faces=None, ks=None, *, dtype=torch.float32, device="cuda", seed=0, offset=0,
                     lo=0.0, offset_add=None, out=None):
    """(X, g): ``n_per_face`` uniform points on each face of the mask ``faces`` (default: all 2d faces) of
    [lo, L_box]^dim, one contiguous block per set bit in increasing bit order, and with ``ks`` the outward normal
    derivative g of the manufactured solution of Poisson_ND.py:49-58 at those points, in one launch
    (pde_sample_faces_rhs).  Point p has the coordinates ``sample_points_rhs`` draws for point p with the same
    seed / offset / offset_add, the block's face coordinate set to lo or L_box.  ``out=(X, g)``: write into existing
    tensors (g may be None)."""
    lib = L.load()
    dev = torch.device(device)
    mask = all_faces(dim) if faces is None else int(faces)
    n = bin(mask).count("1") * int(n_per_face) if 0 < mask < (1 << 2 * dim) else 0
    if out is not None:
        X, g = out
    else:
        X = torch.empty(max(n, 1), dim, dtype=dtype, device=dev)
        g = torch.empty(max(n, 1), dtype=dtype, device=dev) if ks is not None else None
    karr = (C.c_double * dim)(*[float(k) for k in ks]) if ks is not None else None
    with torch.cuda.device(dev):
        L.check(lib.pde_sample_faces_rhs(L.F64 if X.dtype == torch.float64 else L.F32, dim, int(n_per_face), mask, float(lo),
                                         float(L_box), int(seed), int(offset),
                                         offset_add.data_ptr() if offset_add is not None else None, karr, float(L_box),
                                         X.data_ptr(), g.data_ptr() if g is not None else None, _stream(dev)),
                "pde_sample_faces_rhs")
    return X, g


def rank_offset(rank):
    """Philox counter offset of data-parallel rank ``rank``: bits 40.. of the counter's second half, far above any
    epoch count, so that every rank draws its own points (the reference is single-process; with the default seed
    identical draws on every rank would make the global batch n points repeated world times)."""
    return int(rank) << 40


TERMS = ('pde', 'bc', 'data', 'norm')


def _term_weights(weights, rb, has_data, pde=1.0):
    """Weights of the loss terms like the reference's ``weights`` argument (Poisson_ND.py:169-173): bc 1e4 for a soft
    Dirichlet constraint (``rb``), data 1e3 when data points are given, norm 0; ``weights`` overrides them and may
    only name the terms in ``TERMS``."""
    w = {'pde': float(pde), 'bc': 1e4 if rb else 0.0, 'data': 1e3 if has_data else 0.0, 'norm': 0.0}
    if weights:
        unknown = set(weights) - set(TERMS)
        if unknown:
            raise ValueError(f"unknown loss terms {sorted(unknown)}")
        w.update({k: float(v) for k, v in weights.items()})
    return w


class _FacePoints:
    """``n_boundary // (2 dim)`` points on each face of the mask ``faces`` (default: all 2d faces) of [0, L]^dim
    (Poisson_ND.py:225), redrawn into ``X`` by ``draw`` in one launch: a uniform draw in which face k = (coordinate
    k // 2, side k % 2) gets that coordinate set to 0 or L (:133-139), and with ``ks`` the outward normal derivative
    ``g`` of the manufactured solution.  Equal counts per face, so the mean over all face points is the mean of the
    per-face means."""
    KEY = 0x5851F42D4C957F2D   # xor-ed into the seed: the face draws are independent of the interior draws

    def __init__(self, n_boundary, dim, L_box, dtype, device, faces=None, ks=None, key=KEY):
        self.per_face = max(1, int(n_boundary) // (2 * dim))
        self.faces = all_faces(dim) if faces is None else int(faces)
        self.n, self.dim, self.L, self.ks, self.key = bin(self.faces).count("1") * self.per_face, dim, float(L_box), ks, key
        self.X = torch.empty(self.n, dim, dtype=dtype, device=device)
        self.g = torch.empty(self.n, dtype=dtype, device=device) if ks is not None else None

    def draw(self, seed, offset, counter, advance=False):
        """Fresh face points from Philox block ``offset`` + ``counter`` (a device int64 draw counter, incremented
        after the draw when ``advance``)."""
        sample_faces_rhs(self.per_face, self.dim, self.L, self.faces, self.ks, seed=seed ^ self.key, offset=offset,
                         offset_add=counter, out=(self.X, self.g))
        if advance:
            counter.add_(1)
        return self.X


class FusedAdam:
    """Adam over a list of parameter tensors driven by one flat gradient vector (pde_adam_step).
    State tensors mirror torch.optim.Adam's ``exp_avg`` / ``exp_avg_sq`` / ``step``."""

    def __init__(self, params: Sequence[torch.Tensor], lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.params = list(params)
        if not self.params or len(self.params) > 2 * L.MAX_LINEAR + 1:
            raise NotImplementedError("1 .. 17 parameter tensors")
        p0 = self.params[0]
        for p in self.params:
            if not p.is_cuda or p.dtype != p0.dtype or p.device != p0.device or not p.is_contiguous():
                raise ValueError("parameters must be contiguous CUDA tensors of one dtype on one device")
        self.n = sum(p.numel() for p in self.params)
        self.exp_avg = torch.zeros(self.n, dtype=p0.dtype, device=p0.device)
        self.exp_avg_sq = torch.zeros(self.n, dtype=p0.dtype, device=p0.device)
        self.step_count = torch.zeros(1, dtype=torch.int64, device=p0.device)
        self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay

    def config(self, grad_scale=1.0) -> L.Adam:
        c = L.Adam()
        c.dtype = L.F64 if self.params[0].dtype == torch.float64 else L.F32
        c.n_tensors = len(self.params)
        c.lr, c.beta1, c.beta2, c.eps = float(self.lr), float(self.betas[0]), float(self.betas[1]), float(self.eps)
        c.weight_decay, c.grad_scale = float(self.weight_decay), float(grad_scale)
        for i, p in enumerate(self.params):
            c.param[i] = p.data_ptr()
            c.numel[i] = p.numel()
        return c

    def step(self, grad_flat: torch.Tensor, grad_scale=1.0):
        """``grad_flat``: at least ``self.n`` contiguous values in parameters() order."""
        dev = self.params[0].device
        if grad_flat.numel() < self.n or grad_flat.dtype != self.params[0].dtype or not grad_flat.is_contiguous():
            raise ValueError("flat gradient has the wrong size / dtype")
        cfg = self.config(grad_scale)
        with torch.cuda.device(dev):
            L.check(L.load().pde_adam_step(C.byref(cfg), grad_flat.data_ptr(), self.exp_avg.data_ptr(),
                                           self.exp_avg_sq.data_ptr(), self.step_count.data_ptr(), _stream(dev)),
                    "pde_adam_step")


class Adam:
    """``torch.optim.Adam(params, lr, betas, eps, weight_decay)`` for reference-style epochs (``zero_grad -> loss ->
    backward -> step``) at two or three launches of bookkeeping per step instead of torch's ~45: ``step()`` is one
    ``pde_adam_step`` launch over all parameter tensors, fed by one flat gradient vector (same update rule and state as
    ``FusedAdam``).  Where that vector comes from depends on how the gradients were zeroed:

    * ``zero_grad()`` (``set_to_none=True``, torch's default): no launch.  The drop-in losses hand autograd views of
      *one* flat gradient buffer (``ops._Residual`` / ``ops._Jets``), which autograd adopts as ``p.grad`` without
      copying when ``p.grad`` is None; ``step()`` recognises that layout (same storage, consecutive offsets in
      parameter order) and passes the buffer to the kernel as it is.  A second ``backward()`` accumulates into the
      adopted views in place, which keeps the layout; several operator terms inside one ``backward()`` are summed per
      parameter by the autograd engine before they reach ``p.grad`` and are gathered (below).
    * ``zero_grad(set_to_none=False)``: the ``.grad`` tensors are views of the optimiser's own flat buffer, zeroed by
      one fill; autograd adds into them (one small launch per parameter tensor).

    Gradients that arrive in any other layout (other operators, a different parameter order, hooks) are gathered into
    the optimiser's buffer first (one ``torch.cat``; a parameter without gradient counts as zero gradient — torch.optim
    would skip it).  Nothing synchronises, so an epoch can be captured in a ``GraphedEpoch`` as it is (no ``capturable``
    flag needed); the arithmetic is that of torch's default Adam, bias corrections in double (``capturable=True`` keeps
    its step count in float32 and is ~6e-6 per step away from it)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.params = [p for p in params]
        self._opt = FusedAdam(self.params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        p0 = self.params[0]
        self.flat = torch.zeros(self._opt.n, dtype=p0.dtype, device=p0.device)
        self._off = []
        off = 0
        for p in self.params:
            self._off.append(off)
            off += p.numel()
        self.adopted_steps = 0     # steps that took the gradients where autograd left them (no gather, no fill)
        self.gathered_steps = 0

    @property
    def state(self):
        return {"exp_avg": self._opt.exp_avg, "exp_avg_sq": self._opt.exp_avg_sq, "step": self._opt.step_count}

    def _own_view(self, i):
        p, off = self.params[i], self._off[i]
        return self.flat[off:off + p.numel()].view_as(p)

    def zero_grad(self, set_to_none=True):
        if set_to_none:
            for p in self.params:
                p.grad = None
            return
        es = self.flat.element_size()
        for i, p in enumerate(self.params):
            g = p.grad
            if g is None or g.data_ptr() != self.flat.data_ptr() + self._off[i] * es or not g.is_contiguous():
                p.grad = self._own_view(i)
        self.flat.zero_()

    def _flat_grads(self):
        """The gradients as one flat vector without copying, or None if they are not laid out that way."""
        g0 = self.params[0].grad
        if g0 is None:
            return None
        es = g0.element_size()
        st = g0.untyped_storage()
        base = g0.data_ptr()
        for p, off in zip(self.params, self._off):
            g = p.grad
            if (g is None or g.dtype != g0.dtype or not g.is_contiguous() or g.data_ptr() != base + off * es
                    or g.untyped_storage().data_ptr() != st.data_ptr()):
                return None
        if (g0.storage_offset() + self._opt.n) * es > st.nbytes():
            return None
        return g0.as_strided((self._opt.n,), (1,), g0.storage_offset())

    def step(self):
        flat = self._flat_grads()
        if flat is None:
            zero = None
            parts = []
            for i, p in enumerate(self.params):
                if p.grad is None:
                    if zero is None:
                        zero = torch.zeros(max(q.numel() for q in self.params), dtype=self.flat.dtype, device=self.flat.device)
                    parts.append(zero[:p.numel()])
                else:
                    parts.append(p.grad.reshape(-1))
            flat = torch.cat(parts)      # (not into self.flat: some of the parts may be views of it)
            self.gathered_steps += 1
        else:
            self.adopted_steps += 1
        self._opt.step(flat)


class FusedTrainer:
    """The PINN / DRM branch of ``train_poisson_nd`` (Poisson_ND.py:215-241,281-300) with every epoch
    replayed from one CUDA graph: PDE term plus, when their weights are non-zero, the soft Dirichlet
    penalty of ``bc_mode='RB'`` (:224-228, fresh face points every epoch), the data term (:230-234) and
    the norm term (:236-237); total gradient = sum of weight x term gradient, then Adam.

    model      SolutionNet-style module on a CUDA device (parameters updated in place)
    method     'PINN' | 'DRM'
    X, f       fixed interior points and right-hand side; default: drawn once like the reference
               (:193-194), or every epoch with ``resample=True`` (what the WAN branch does, :246,:256)
    weights    {'pde','bc','data','norm'} like the reference's ``weights`` argument; defaults follow :169-173
               (bc 1e4 for an 'RB' model, data 1e3 when data points are given, norm 0)
    n_boundary face points per epoch, split evenly over the 2d faces (:225)
    X_data, u_data   fixed data points / values (:197-202)
    norm_mode  'nontrivial' (1 / (mean u^2 + 1e-8)) | 'l2' (mean u^2) on the interior points (:143-147)
    n_test     > 0: L2 evaluation on freshly drawn test points after each step and device-side
               best-parameter tracking (:281-300)
    history    number of epochs whose loss (and L2) are kept in device arrays (0: none)
    group      data parallelism over points: every rank runs the same epoch on its own points (the rank selects
               the sampler's Philox counter block, ``rank_offset``) and the
               [grad | dE | sums] rows are summed over the ranks before Adam (exchange='nvlink': one kernel over
               peer memory; 'nccl': torch.distributed.all_reduce)
    neumann_faces    face mask (face k = side k % 2 of axis k // 2, ``all_faces(dim)`` for every face) on which the
               Neumann condition du/dn = du*/dn of the manufactured solution is imposed as the penalty term
               mean((du/dn - g)^2), weight ``weight_neumann``, reported as ``terms['neumann']``: fresh face points every
               epoch, n_boundary // (2d) per face, g from the same launch.  The Dirichlet ``bc`` penalty then covers the
               other faces only.  Needs an 'RB' model (the 'FBC' envelope forces u = 0 on every face).
    robin_kappa      kappa of the Robin condition du/dn + kappa u = g on the ``neumann_faces`` (0: Neumann), in either
               form; g = du*/dn + kappa u* on the face points (u* from one sample_points_rhs launch on those points)
    neumann_form     'penalty': the row above (PROG_FLUX, beta = kappa); 'ritz' (method='DRM' only): the boundary term
               of the Deep Ritz functional, mean(kappa u^2 / 2 - g u) on the same face points (PROG_RITZ_VALUE), with
               the weight the functional fixes, the pde weight * popcount(neumann_faces) / L (DESIGN.md §3.4b);
               ``weight_neumann`` (default 1) is for the penalty form only
    mean_value       add the row 'mean' = (mean_X u - c*)^2 on the interior points, weight ``weight_mean``, with c* the
               exact mean of u* over the box: it fixes the additive constant of a pure-Neumann problem
               (``neumann_faces=all_faces(dim)``).  Not available with ``group``.
    """

    TERMS = TERMS
    NEUMANN_KEY = 0x2545F4914F6CDD1D   # xor-ed into the seed: the Neumann face draws are independent of the others

    def __init__(self, model, L_box=2.0, ks=None, method='PINN', n_interior=20000, lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                 weight_pde=1.0, X=None, f=None, resample=False, seed=0, n_test=0, history=0, graph=True, group=None,
                 envelope: Optional[EnvelopeSpec] = None, exchange='nvlink', weights=None, n_boundary=4000, X_data=None,
                 u_data=None, norm_mode='nontrivial', neumann_faces=None, weight_neumann=None, neumann_form='penalty',
                 robin_kappa=0.0, mean_value=False, weight_mean=1.0):
        from .poisson import _envelope
        self.lib = L.load()
        self.model, self.L, self.method, self.group = model, float(L_box), method, group
        p0 = next(model.parameters())
        self.dev, self.dtype = p0.device, p0.dtype
        if method not in ('PINN', 'DRM'):
            raise ValueError("method must be one of {'PINN','DRM'}")
        if neumann_form not in ('penalty', 'ritz'):
            raise ValueError("neumann_form must be 'penalty' or 'ritz'")
        if neumann_form == 'ritz':
            if method != 'DRM' or neumann_faces is None:
                raise ValueError("neumann_form='ritz' is the boundary term of the Deep Ritz functional: it needs "
                                 "method='DRM' and neumann_faces")
            if weight_neumann is not None:
                raise ValueError("the Ritz boundary term has the weight the functional fixes; weight_neumann is for "
                                 "neumann_form='penalty'")
        if mean_value and group is not None:
            raise NotImplementedError("the mean-value constraint is a function of a global mean: not available with "
                                      "group")
        if norm_mode not in ('nontrivial', 'l2'):
            raise ValueError("norm mode should be 'nontrivial' or 'l2'")
        self.env = envelope if envelope is not None else _envelope(model, L_box)
        self.spec = ProgramSpec(L.PROG_PINN, alpha=-1.0) if method == 'PINN' else ProgramSpec(L.PROG_DRM, alpha=0.5)
        self.dim = getattr(model, "dim", None) or _Net(model, torch.empty(1, 1, device=self.dev, dtype=self.dtype)).dim
        self.ks = [1.0] * self.dim if ks is None else [float(k) for k in ks]
        self.seed, self.resample = int(seed), bool(resample)
        self.world, self.rank = 1, 0
        if group is not None:
            import torch.distributed as dist
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if X is None:
            self.n = int(n_interior)
            self.X, _, self.f = sample_points_rhs(self.n, self.dim, self.L, self.ks, dtype=self.dtype, device=self.dev,
                                                  seed=self.seed, offset=rank_offset(self.rank))
        else:
            self.X = X.detach().to(self.dtype).contiguous()
            self.n = self.X.shape[0]
            self.f = (f if f is not None else sample_points_rhs(0, 0, self.L, self.ks, X=self.X)[2]).detach().to(self.dtype).reshape(-1).contiguous()
            if self.resample:
                raise ValueError("resample=True draws its own points; do not pass X")
        rb = getattr(model, "bc_mode", "FBC") == 'RB' and envelope is None
        self.w = _term_weights(weights, rb, X_data is not None, pde=weight_pde)
        self.norm_mode = norm_mode
        self.neumann_faces = None if neumann_faces is None else int(neumann_faces)
        dirichlet_faces = all_faces(self.dim)
        if self.neumann_faces is not None:
            if not rb:
                raise ValueError("neumann_faces needs an 'RB' model without envelope: the 'FBC' envelope forces u = 0 "
                                 "on every face")
            if not 0 < self.neumann_faces < all_faces(self.dim) + 1:
                raise ValueError(f"neumann_faces must be a face mask in 1 .. {all_faces(self.dim)}")
            dirichlet_faces &= ~self.neumann_faces
            if neumann_form == 'ritz':    # the boundary integral over |Omega|: popcount faces of area L^(d-1) / L^d
                self.w['neumann'] = self.w['pde'] * bin(self.neumann_faces).count("1") / self.L
            else:
                self.w['neumann'] = 1.0 if weight_neumann is None else float(weight_neumann)
        self.neumann_form, self.kappa = neumann_form, float(robin_kappa)
        if mean_value:
            self.w['mean'] = float(weight_mean)
            # c* = mean of u* = prod_i sin(k_i pi x_i / L) over [0, L]^d
            self.c_mean = math.prod((1.0 - math.cos(k * math.pi)) / (k * math.pi) for k in self.ks)
        self.use = {'pde': True, 'bc': self.w['bc'] != 0.0 and dirichlet_faces != 0, 'data': self.w['data'] != 0.0,
                    'norm': self.w['norm'] > 0.0, 'neumann': self.neumann_faces is not None, 'mean': bool(mean_value)}
        if self.use['data'] and (X_data is None or u_data is None):
            raise ValueError("a data weight needs X_data and u_data")
        if self.use['norm'] and norm_mode == 'nontrivial' and group is not None:
            raise NotImplementedError("the 'nontrivial' norm term is a function of a global mean: not available with group "
                                      "(use norm_mode='l2' or weight 0)")
        self.rows = [t for t in self.TERMS + ('neumann', 'mean') if self.use[t]]
        self.net = _Net(model, self.X)
        self.params = [p for p in self.net.params]
        self.nparam = sum(p.numel() for p in self.params)
        self.opt = FusedAdam([p.data for p in self.params], lr=lr, betas=betas, eps=eps)
        self._ar = None
        # one row per active term: [grad (nparam) | dE (1) | sum (1)] — the layout pde_residual_loss_grad writes
        self.G = torch.zeros(len(self.rows), self.nparam + 2, dtype=self.dtype, device=self.dev)
        if group is not None:
            if exchange == 'nvlink':     # one-kernel all-reduce over peer memory (pde_allreduce_oneshot)
                from .comm import NvlinkAllReduce
                self._ar = NvlinkAllReduce(group, self.G.numel(), self.dtype, self.dev)
            elif exchange != 'nccl':
                raise ValueError("exchange must be 'nvlink' or 'nccl'")
        if len(self.rows) > 1:
            self.total = torch.zeros(self.nparam + 2, dtype=self.dtype, device=self.dev)
            self.wvec = torch.tensor([self.w[t] for t in self.rows], dtype=self.dtype, device=self.dev)
        if self.use['bc']:
            self.faces = _FacePoints(n_boundary, self.dim, self.L, self.dtype, self.dev, faces=dirichlet_faces)
            self.nb, self.Xb = self.faces.n, self.faces.X
        if self.use['neumann']:
            self.nfaces = _FacePoints(n_boundary, self.dim, self.L, self.dtype, self.dev, faces=self.neumann_faces,
                                      ks=self.ks, key=self.NEUMANN_KEY)
            self.nn, self.Xn, self.gn = self.nfaces.n, self.nfaces.X, self.nfaces.g
            if neumann_form == 'ritz':
                self.nspec = ProgramSpec(L.PROG_RITZ_VALUE, alpha=0.0, beta_const=self.kappa)
            else:
                self.nspec = ProgramSpec(L.PROG_FLUX, alpha=1.0, beta_const=self.kappa, faces=self.neumann_faces)
            if self.kappa != 0.0:
                self.un = torch.empty(self.nn, dtype=self.dtype, device=self.dev)    # u* on the face points
        if self.use['data']:
            self.Xd = X_data.detach().to(self.dtype).to(self.dev).contiguous()
            self.ud = u_data.detach().to(self.dtype).to(self.dev).reshape(-1).contiguous()
        if self.use['norm']:
            self.nsum = torch.zeros(1, dtype=self.dtype, device=self.dev)
            self.nseed = torch.ones(1, dtype=self.dtype, device=self.dev)
            self.norm_value = torch.zeros((), dtype=self.dtype, device=self.dev)
        if self.use['mean']:
            self.msum = torch.zeros(1, dtype=self.dtype, device=self.dev)
            self.mseed = torch.ones(1, dtype=self.dtype, device=self.dev)
            self.mean_term = torch.zeros((), dtype=self.dtype, device=self.dev)
            self.mspec = ProgramSpec(L.PROG_RITZ_VALUE, alpha=-1.0)     # q = u
        self.n_test = int(n_test)
        if self.n_test:
            self.Xt = torch.empty(self.n_test, self.dim, dtype=self.dtype, device=self.dev)
            self.ut = torch.empty(self.n_test, dtype=self.dtype, device=self.dev)
            self.esum = torch.zeros(1, dtype=self.dtype, device=self.dev)
            self.best_metric = torch.full((1,), float("inf"), dtype=self.dtype, device=self.dev)
            self.best_flat = torch.zeros(self.nparam, dtype=self.dtype, device=self.dev)
            self.best_step = torch.full((1,), -1, dtype=torch.int64, device=self.dev)
        self.hist_loss = torch.zeros(max(int(history), 0), dtype=self.dtype, device=self.dev)
        self.hist_l2sq = torch.zeros(max(int(history), 0) if self.n_test else 0, dtype=self.dtype, device=self.dev)
        self._order = self.lib.pde_program_order(self.spec.kind)
        cnet = self.net.to_c([p.data for p in self.params])
        n_big = max(self.n, self.n_test, getattr(self, "nb", 1), getattr(self, "nn", 1),
                    self.Xd.shape[0] if self.use['data'] else 1)
        self._ws = _ws_for(cnet, self._order, n_big, self.dev)
        self._graph = None
        self._use_graph = bool(graph)
        self.epochs_done = 0

    # ---- the launches of one epoch (enqueued on the current stream, no host sync)
    def _mse(self, cnet, cenv, X, target, term, seed=None, sums=None, want_grad=True):
        """mean((u - target)^2) over the global batch (target None: mean u^2) into the row of ``term``."""
        n = X.shape[0]
        _residual_row(cnet, cenv, _MSE.to_c(f=target), X, n, 1.0 / (n * self.world), self._ws,
                      self.G[self.rows.index(term)], self.nparam, seed=seed, sums=sums, want_grad=want_grad)

    def _enqueue(self):
        cnet = self.net.to_c([p.data for p in self.params])
        cenv = self.env.to_c()
        P, step = self.nparam, self.opt.step_count
        if self.resample:
            sample_points_rhs(self.n, self.dim, self.L, self.ks, dtype=self.dtype, device=self.dev, seed=self.seed,
                              offset=rank_offset(self.rank), offset_add=step, out=(self.X, None, self.f))
        inv_n = 1.0 / (self.n * self.world)
        row = self.rows.index('pde')
        # a single row: its exchange folded into the reduction of the per-CTA partials (one launch fewer)
        fused_ar = self._ar if len(self.rows) == 1 else None
        _residual_row(cnet, cenv, self.spec.to_c(f=self.f), self.X, self.n, inv_n, self._ws, self.G[row], P, ar=fused_ar)
        if self.use['bc']:
            self._mse(cnet, cenv, self.faces.draw(self.seed, rank_offset(self.rank), step), None, 'bc')
        if self.use['data']:
            self._mse(cnet, cenv, self.Xd, self.ud, 'data')
        if self.use['neumann']:
            self.nfaces.draw(self.seed, rank_offset(self.rank), step)
            if self.kappa != 0.0:     # g = du*/dn + kappa u*
                sample_points_rhs(0, 0, self.L, self.ks, X=self.Xn, out=(None, self.un, None))
                self.gn.add_(self.un, alpha=self.kappa)
            _residual_row(cnet, cenv, self.nspec.to_c(f=self.gn), self.Xn, self.nn, 1.0 / (self.nn * self.world), self._ws,
                          self.G[self.rows.index('neumann')], P)
        if self.use['norm']:
            if self.norm_mode == 'l2':
                self._mse(cnet, cenv, self.X, None, 'norm')
            else:
                # F = 1 / (m + 1e-8), m = mean u^2: the mean first, then the reverse sweep seeded with dF/dm
                self._mse(cnet, cenv, self.X, None, 'norm', sums=self.nsum, want_grad=False)
                m = self.nsum * inv_n
                torch.neg(torch.reciprocal((m + 1e-8) ** 2), out=self.nseed)
                self._mse(cnet, cenv, self.X, None, 'norm', seed=self.nseed)
                self.norm_value.copy_(torch.reciprocal(m + 1e-8)[0])
        if self.use['mean']:
            # (m - c*)^2, m = mean u: the mean first, then the reverse sweep seeded with 2 (m - c*)
            row_m = self.G[self.rows.index('mean')]
            _residual_row(cnet, cenv, self.mspec.to_c(), self.X, self.n, inv_n, self._ws, None, P, sums=self.msum,
                          want_grad=False)
            dm = self.msum * inv_n - self.c_mean
            torch.mul(dm, 2.0, out=self.mseed)
            _residual_row(cnet, cenv, self.mspec.to_c(), self.X, self.n, inv_n, self._ws, row_m, P, seed=self.mseed)
            self.mean_term.copy_((dm * dm)[0])
        if self._ar is not None:
            if fused_ar is None:
                self._ar.all_reduce_(self.G.view(-1))
        elif self.group is not None:
            import torch.distributed as dist
            dist.all_reduce(self.G, group=self.group)
        if self.hist_loss.numel():
            self.hist_loss.index_copy_(0, step.clamp(max=self.hist_loss.numel() - 1), _row_sums(self.G[row], P) * inv_n)
        if len(self.rows) > 1:
            torch.mv(self.G.t(), self.wvec, out=self.total)      # sum of weight x term gradient
            self.opt.step(self.total)
        else:
            self.opt.step(self.G[0], self.w['pde'])
        if self.n_test:
            # fresh test points every epoch (Poisson_ND.py:282), a different Philox key than the interior draw
            sample_points_rhs(self.n_test, self.dim, self.L, self.ks, dtype=self.dtype, device=self.dev,
                              seed=self.seed ^ 0x9E3779B97F4A7C15, offset_add=step, out=(self.Xt, self.ut, None))
            _residual_row(cnet, cenv, _MSE.to_c(f=self.ut), self.Xt, self.n_test, 1.0 / self.n_test, self._ws, None, P,
                          sums=self.esum, want_grad=False)
            L.check(self.lib.pde_keep_best(C.byref(self.opt.config()), self.esum.data_ptr(), self.best_metric.data_ptr(),
                                           self.best_flat.data_ptr(), step.data_ptr(), self.best_step.data_ptr(),
                                           _stream(self.dev)), "pde_keep_best")
            if self.hist_l2sq.numel():
                self.hist_l2sq.index_copy_(0, (step - 1).clamp(min=0, max=self.hist_l2sq.numel() - 1),
                                           self.esum / self.n_test)

    def step(self, n_epochs=1):
        """Run ``n_epochs`` epochs (graph replays after the first call)."""
        with torch.cuda.device(self.dev):
            for _ in range(int(n_epochs)):
                if not self._use_graph:
                    self._enqueue()
                elif self._graph is None:
                    # warm-up epoch outside the graph (module loading, cudaFuncSetAttribute), then capture
                    self._enqueue()
                    torch.cuda.synchronize(self.dev)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._enqueue()
                    self._graph = g
                    self.epochs_done += 1
                    continue
                else:
                    self._graph.replay()
                self.epochs_done += 1
        return self

    # ---- read-backs (these synchronise)
    def check(self):
        """Raise if the NVLink exchange ever timed out on this rank (synchronises the stream)."""
        if self._ar is not None:
            self._ar.check()

    def _mean(self, term, n):
        """The mean over the global batch of ``n`` points per rank that the row of ``term`` holds."""
        return _row_sums(self.G[self.rows.index(term)], self.nparam)[0] / (n * self.world)

    @property
    def loss(self):
        """PDE loss of the last evaluated epoch (mean over the global batch), 0-d device tensor."""
        self.check()
        return self._mean('pde', self.n)

    @property
    def terms(self):
        """{'pde','bc','data','norm','total'} (and 'neumann' with ``neumann_faces``: the row's mean in either form,
        'mean' with ``mean_value``) of the last evaluated epoch as 0-d device tensors (what train_poisson_nd appends to
        its history, Poisson_ND.py:288-293); 'total' includes every term with its weight."""
        self.check()
        out = {t: torch.zeros((), dtype=self.dtype, device=self.dev) for t in self.TERMS}
        out['pde'] = self._mean('pde', self.n)
        if self.use['bc']:
            out['bc'] = self._mean('bc', self.nb)
        if self.use['data']:
            out['data'] = self._mean('data', self.Xd.shape[0])
        if self.use['norm']:
            out['norm'] = self._mean('norm', self.n) if self.norm_mode == 'l2' else self.norm_value
        out['total'] = sum(self.w[t] * out[t] for t in self.TERMS)
        if self.use['neumann']:
            out['neumann'] = self._mean('neumann', self.nn)
            out['total'] = out['total'] + self.w['neumann'] * out['neumann']
        if self.use['mean']:
            out['mean'] = self.mean_term
            out['total'] = out['total'] + self.w['mean'] * out['mean']
        return out

    @property
    def l2(self):
        """L2 error on the last test draw: sqrt(mean((u - u*)^2))   (Poisson_ND.py:285)."""
        if not self.n_test:
            raise ValueError("constructed with n_test=0")
        return (self.esum[0] / self.n_test).sqrt()

    @property
    def best_l2(self):
        return (self.best_metric[0] / self.n_test).sqrt()

    def load_best(self, model=None):
        """Copy the best parameters seen so far into ``model`` (default: the trained model)."""
        tgt = self.params if model is None else _Net(model, self.X).params
        with torch.no_grad():
            for p, b in zip(tgt, _split_flat(self.best_flat, tgt)):
                p.copy_(b)


class WanTrainer:
    """The WAN branch of ``train_poisson_nd`` (Poisson_ND.py:242-276): per epoch ``critic_steps`` critic updates on
    freshly drawn interior points (``loss_v`` of wan_losses, :244-248), then one solution update on another fresh draw
    with ``w_pde loss_pde_u + w_bc bc + w_data data + w_norm norm`` (:251-271).  The losses are the drop-in operators
    of ``pde_b200.poisson`` (both networks' jets and reverse sweeps on the fused kernels), the optimisers are
    ``pde_b200.train.Adam`` (torch.optim.Adam's arithmetic, one launch per step), the points come from the device
    sampler with a draw counter, and the whole epoch is captured into one CUDA graph (``graph=True``).

    ``record_points=True`` (eager mode only) keeps every draw in ``self.drawn`` = [(kind, X, f) ...] so that a
    reference loop can be run on identical points.
    """

    def __init__(self, model, critic, L_box=2.0, ks=None, n_interior=20000, lr=1e-3, critic_steps=3, wan_reg=1.0,
                 weights=None, n_boundary=4000, X_data=None, u_data=None, norm_mode='nontrivial', seed=0, graph=True,
                 record_points=False):
        from . import poisson as P
        self.P = P
        self.model, self.critic, self.L = model, critic, float(L_box)
        p0 = next(model.parameters())
        self.dev, self.dtype = p0.device, p0.dtype
        self.dim = model.dim
        self.ks = [1.0] * self.dim if ks is None else [float(k) for k in ks]
        self.n, self.critic_steps, self.wan_reg = int(n_interior), int(critic_steps), float(wan_reg)
        self.w = _term_weights(weights, getattr(model, "bc_mode", "FBC") == 'RB', X_data is not None)
        self.norm_mode = norm_mode
        self.seed = int(seed)
        self.opt_u = Adam(model.parameters(), lr=lr)      # torch.optim.Adam's update, one launch per step
        self.opt_v = Adam(critic.parameters(), lr=lr)
        self.u_params, self.v_params = list(model.parameters()), list(critic.parameters())
        self.draws = torch.zeros(1, dtype=torch.int64, device=self.dev)
        # static point buffers (one per evaluation of the epoch, so that the autograd graphs of an epoch do not alias)
        mk = lambda n: (torch.empty(n, self.dim, dtype=self.dtype, device=self.dev).requires_grad_(True), None,
                        torch.empty(n, 1, dtype=self.dtype, device=self.dev))
        self.bufs = [mk(self.n) for _ in range(self.critic_steps + 1)]
        if self.w['bc'] != 0.0:
            self.faces = _FacePoints(n_boundary, self.dim, self.L, self.dtype, self.dev)
        self.Xd = X_data.detach().to(self.dev, self.dtype).contiguous() if X_data is not None else None
        self.ud = u_data.detach().to(self.dev, self.dtype).contiguous() if u_data is not None else None
        self.record = bool(record_points) and not graph
        self.drawn = []
        self._ep = GraphedEpoch(self._epoch, device=self.dev) if graph else None
        self.last = None

    def _draw(self, buf, kind):
        X, _, f = buf
        sample_points_rhs(self.n, self.dim, self.L, self.ks, dtype=self.dtype, device=self.dev, seed=self.seed,
                          offset_add=self.draws, out=(X.detach(), None, f))
        self.draws.add_(1)
        if self.record:
            self.drawn.append((kind, X.detach().clone(), f.clone()))
        return X, f

    def _epoch(self):
        P = self.P
        loss_v = None
        for k in range(self.critic_steps):                                   # Poisson_ND.py:244-248
            X, f = self._draw(self.bufs[k], 'v')
            _, loss_v, _, _ = P.wan_losses(self.model, self.critic, X, f, self.L, v_reg_weight=self.wan_reg)
            self.opt_v.zero_grad()
            loss_v.backward(inputs=self.v_params)
            self.opt_v.step()
        X, f = self._draw(self.bufs[self.critic_steps], 'u')                 # :251-253
        loss_pde_u, _, weak, phi_n = P.wan_losses(self.model, self.critic, X, f, self.L, v_reg_weight=self.wan_reg)
        zero = torch.zeros((), dtype=self.dtype, device=self.dev)
        bc_l = data_l = norm_l = zero
        if self.w['bc'] != 0.0:                                              # :255-259 on device-drawn face points
            Xb = self.faces.draw(self.seed, 0, self.draws, advance=True)
            if self.record:
                self.drawn.append(('bc', Xb.clone(), None))
            bc_l = P.data_loss(self.model, Xb, None, self.L)
        if self.w['data'] != 0.0:                                            # :261-265
            data_l = P.data_loss(self.model, self.Xd, self.ud, self.L)
        if self.w['norm'] > 0.0:                                             # :267-268
            norm_l = P.norm_loss(P.solution_jets(self.model, X.detach(), self.L, 0)[0], mode=self.norm_mode)
        loss = self.w['pde'] * loss_pde_u + self.w['bc'] * bc_l + self.w['data'] * data_l + self.w['norm'] * norm_l
        self.opt_u.zero_grad()
        loss.backward(inputs=self.u_params)
        self.opt_u.step()
        return {'total': loss.detach(), 'pde': loss_pde_u.detach(), 'bc': bc_l.detach(), 'data': data_l.detach(),
                'norm': norm_l.detach(), 'wan_loss_v': loss_v.detach() if loss_v is not None else zero,
                'wan_weak': weak, 'wan_phi_norm': phi_n}

    def step(self, n_epochs=1):
        for _ in range(int(n_epochs)):
            self.last = self._ep() if self._ep is not None else self._epoch()
        return self


class GraphedEpoch:
    """Capture a reference-style epoch — ``zero_grad -> losses -> backward -> optimizer.step`` written
    against the drop-in loss functions — into one CUDA graph and replay it.

    The drop-in operators enqueue everything on the current stream and never synchronise, so the host
    side of an epoch (Python, autograd bookkeeping, ~20 small launches per loss) disappears on replay;
    this is what makes the latency-bound configurations (1 000 – 40 000 points: IPW / QHO / KH grids,
    BASELINE.json configs 1, 4, 5) run at kernel speed.  Requirements on ``fn``: static input tensors,
    no ``.item()`` / host read-back inside, optimisers built with ``capturable=True`` (or ``pb.train.Adam``, which
    updates all parameter tensors in one launch), gradients allocated before capture (``warmup`` eager epochs on a
    side stream take care of that).

        opt = torch.optim.Adam(model.parameters(), lr=1e-3, capturable=True)
        def epoch():
            opt.zero_grad(set_to_none=False)
            loss = I.PINN_loss(model, x, n, L); loss.backward(); opt.step()
            return loss
        ep = pb.train.GraphedEpoch(epoch); ep(); ...; print(float(ep.out))
    """

    def __init__(self, fn, warmup=3, device=None):
        self.fn = fn
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.graph = None
        self.out = None
        self.warmup = int(warmup)
        self.replays = 0

    def _capture(self):
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                self.out = self.fn()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.out = self.fn()
        self.graph = g

    def __call__(self):
        """Run one epoch; returns ``fn``'s output tensors (static storage, overwritten by every replay).
        The first call runs ``warmup`` eager epochs and captures; it does not replay, so that the number
        of optimiser steps taken equals ``warmup`` after it (then +1 per call)."""
        with torch.cuda.device(self.dev):
            if self.graph is None:
                self._capture()
            else:
                self.graph.replay()
                self.replays += 1
        return self.out
